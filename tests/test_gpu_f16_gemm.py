"""fp16 / bf16 tensor-core GEMMs of csrc/igemm_tc.cu (fpcc_spconv_f16, fpcc_linear_f16 dense and selection form,
fpcc_spconv_wgrad_f16) against the fp64 oracle of tests/f16_gemm_oracle.py, at the shapes where these kernels go wrong:
K tails of 8 channels, several 256-column blocks, column counts that are not multiples of 8 or 16, more than 27 and more
than 28 kernel offsets (no neighbour prefetch; three operand stages), tiles without any active offset, empty selection
groups, and more 128-row tiles than SMs, so that every CTA reuses its TMEM accumulator slots and metadata slots.

(a) Integer-exact.  Inputs and weights are small integers, exact in fp16 and bf16; biases are distinct integers per
    column; residuals are integers; LeakyReLU slopes are 1/4 and 1/2.  Every product is exact in fp32 and every partial
    sum is an integer or a dyadic rational of a few bits below 2^24 (the oracle asserts sum |terms| < 2^20 per output
    element), so fp32 accumulation is exact in any order, rounded to nearest or truncated.  The fp32 output must then
    equal the fp64 reference bit for bit, and an fp16 / bf16 output its single round-to-nearest cast.  This is reasoning
    about the tcgen05 accumulator, not a measurement.
(b) Error bound on random data: |got - ref| <= 2 n 2^-24 S per element (n = kvol C_in + 3, S = sum |a w| + |b| + |res|),
    the textbook worst case of fp32 summation in any order with truncation allowed.  Catches a reduced-precision
    accumulator or a bias added after a rounding, which integers cannot show.  fp16 / bf16 outputs equal the
    round-to-nearest cast of the fp32-output launch (same instance, same accumulation order), overflow to +-inf included.
(c) Invariances, bit-exact: the same launch twice, the SM budget (one CTA walking every tile), a random row_perm.
(d) The weight gradient, integer-exact, at every pair-count edge of its 64-pair stages and 2048-pair tiles.
(e) One case with byte offsets beyond 2^31 in the input and the output."""
import numpy as np
import pytest
import torch

from tests import f16_gemm_oracle as FO

pytestmark = pytest.mark.gpu

F16, BF16, F32 = torch.float16, torch.bfloat16, torch.float32
_DT = {F16: 0, BF16: 1}
_OT = {F16: 0, BF16: 1, F32: 2}
IO = [(F16, F16), (F16, BF16), (F16, F32), (BF16, F16), (BF16, BF16), (BF16, F32)]  # (inputs, output)
_NAME = {F16: 'f16', BF16: 'bf16', F32: 'f32'}
SLOPE, POST_SLOPE = 0.25, 0.5


def _lib():
    from fastpcc_b200 import _lib as L
    return L


def _p(t):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _gen(seed):
    return torch.Generator(device='cuda').manual_seed(seed)


def _ints(shape, r, dtype, g):
    return torch.randint(-r, r + 1, shape, generator=g, device='cuda', dtype=torch.int32).to(dtype)


def _conv(f, w_t, tbuf, n_out, bias=None, code=FO.ACT_NONE, slope=0.0, res=None, post=FO.ACT_NONE, post_slope=0.0,
          out_dtype=F32, row_perm=None):
    """fpcc_spconv_f16 through the C ABI; tbuf is the k-major table [kvol, ld] (ld >= n_out)"""
    kv, co, ci = w_t.shape
    out = torch.empty((n_out, co), dtype=out_dtype, device='cuda')
    _lib().call('fpcc_spconv_f16', _p(f), _DT[f.dtype], f.shape[0], ci, _p(w_t), kv, co, _p(tbuf), tbuf.shape[1], n_out,
                _p(row_perm), _p(bias), code, slope, _p(res), post, post_slope, _p(out), _OT[out_dtype], _stream())
    return out


def _linear(a, w, bias=None, code=FO.ACT_NONE, slope=0.0, res=None, post=FO.ACT_NONE, post_slope=0.0, out_dtype=F32,
            sel=None, out=None):
    """fpcc_linear_f16 through the C ABI; sel = (sel_row, sel_out, offsets [n_groups + 1]) writes into `out`"""
    m, k = a.shape
    if sel is None:
        n = w.shape[0]
        out = torch.empty((m, n), dtype=out_dtype, device='cuda')
        _lib().call('fpcc_linear_f16', _p(a), _DT[a.dtype], m, k, _p(w), n, None, None, None, 1, 0, _p(bias), code, slope,
                    _p(res), post, post_slope, _p(out), _OT[out_dtype], _stream())
        return out
    sel_row, sel_out, offsets = sel
    groups = offsets.numel() - 1
    n = w.shape[0] // groups
    _lib().call('fpcc_linear_f16', _p(a), _DT[a.dtype], m, k, _p(w), n, _p(sel_row), _p(sel_out), _p(offsets), groups,
                sel_out.numel(), _p(bias), code, slope, _p(res), post, post_slope, _p(out), _OT[out.dtype], _stream())
    return out


def _assert_bits(got, want, what=''):
    """bit-identical, except that +0 and -0 count as equal"""
    assert got.shape == want.shape and got.dtype == want.dtype, (got.shape, want.shape, got.dtype, want.dtype)
    iv = torch.int32 if got.dtype == F32 else torch.int16
    same = (got.view(iv) == want.view(iv)) | ((got == 0) & (want == 0))
    if not bool(same.all()):
        bad = torch.nonzero(~same)
        r, c = (int(v) for v in bad[0])
        raise AssertionError(f'{what}: {bad.shape[0]} of {got.numel()} elements differ; first at row {r}, column {c}: '
                             f'got {float(got[r, c])!r}, want {float(want[r, c])!r} (rows with a mismatch: '
                             f'{torch.unique(bad[:, 0]).numel()}, columns: {torch.unique(bad[:, 1]).tolist()[:16]})')


def _epi(epi, idx):
    """epilogue level 0..7: bit 0 act (LeakyReLU 1/4 or ReLU, by case), bit 1 residual, bit 2 post act (LeakyReLU 1/2)"""
    code = (FO.ACT_LEAKY if idx % 2 == 0 else FO.ACT_RELU) if epi & 1 else FO.ACT_NONE
    post = FO.ACT_LEAKY if epi & 4 else FO.ACT_NONE
    return code, bool(epi & 2), post


def _int_bias(n, g, idx):
    """distinct integers per column (a bias read from the wrong column block cannot go unseen); none in every 5th case"""
    if idx % 5 == 4:
        return None
    return (torch.randperm(n, generator=g, device='cuda') - n // 2).to(F32)


# ---- (a) integer-exact matrix --------------------------------------------------------------------------------------------
C_IN = (16, 24, 40, 64, 72, 128, 136, 256, 264, 512)
C_OUT = (16, 17, 20, 24, 40, 48, 100, 128, 255, 256, 257, 300, 512)
KVOL = (1, 2, 8, 27, 28, 32)
N_OUT = (1, 127, 128, 129, 45000)  # 45000 rows: 352 tiles, 2-3 per CTA on 148 SMs (4-7 with two column blocks)
CONV_CASES = FO.pairwise([C_IN, C_OUT, KVOL, N_OUT, tuple(range(len(IO))), tuple(range(8)), FO.BUILDERS], seed=1) + [
    (64, 256, 32, 45000, 2, 7, 'random'),      # three operand stages (kvol >= 29 at n_tile 256), many tiles per CTA
    (128, 300, 29, 3000, 5, 3, 'empty_tile'),  # three stages, two column blocks
    (136, 256, 28, 2000, 0, 5, 'one_row'),     # the largest kvol with four stages
    (512, 512, 32, 45000, 2, 6, 'dense'),      # every K stage and column block full
    (24, 17, 27, 45000, 4, 1, 'empty_tile'),   # prefetched neighbours, scalar stores, empty tiles at many CTA slots
    (16, 20, 32, 45000, 3, 2, 'one_row'),      # no prefetch, offset masks only in the OR over warps
    (264, 257, 1, 129, 1, 7, 'edge'),
]


def _conv_id(c):
    ci, co, kv, n, io, epi, kind = c
    return f'ci{ci}-co{co}-kv{kv}-n{n}-{_NAME[IO[io][0]]}to{_NAME[IO[io][1]]}-e{epi}-{kind}'


@pytest.mark.parametrize('case', CONV_CASES, ids=[_conv_id(c) for c in CONV_CASES])
def test_spconv_f16_integer_exact(case):
    ci, co, kv, n_out, io, epi, kind = case
    idx = CONV_CASES.index(case)
    dt, ot = IO[io]
    g = _gen(1000 + idx)
    n_in = max(n_out, 300) + 3
    f = _ints((n_in, ci), 8, dt, g)
    w_t = _ints((kv, co, ci), 8, dt, g)
    table = FO.build_table(kind, kv, n_out, n_in, seed=idx).cuda()
    ld = n_out + 8 * (idx % 3)  # row pitch above n_out in two cases of three; the spare columns must not be read
    tbuf = torch.ones((kv, ld), dtype=torch.int32, device='cuda')
    tbuf[:, :n_out] = table
    bias = _int_bias(co, g, idx)
    code, has_res, post = _epi(epi, idx)
    res = _ints((n_out, co), 64, ot, g) if has_res else None
    got = _conv(f, w_t, tbuf, n_out, bias, code, SLOPE, res, post, POST_SLOPE, ot)
    FO.assert_exact_premise(FO.abs_sum(f, w_t, table, bias, res))
    want = FO.spconv(f, w_t, table, bias, code, SLOPE, res, post, POST_SLOPE).float().to(ot)
    _assert_bits(got, want, _conv_id(case))


M_LIN = (1, 128, 129, 3000, 40000)
K_LIN = (16, 24, 200, 1024, 2048)
N_LIN = (16, 20, 64, 256, 264, 512, 1024)
LIN_CASES = FO.pairwise([M_LIN, K_LIN, N_LIN, tuple(range(len(IO))), tuple(range(8))], seed=2)


def _lin_id(c):
    m, k, n, io, epi = c
    return f'm{m}-k{k}-n{n}-{_NAME[IO[io][0]]}to{_NAME[IO[io][1]]}-e{epi}'


@pytest.mark.parametrize('case', LIN_CASES, ids=[_lin_id(c) for c in LIN_CASES])
def test_linear_f16_integer_exact(case):
    m, k, n, io, epi = case
    idx = LIN_CASES.index(case)
    dt, ot = IO[io]
    g = _gen(2000 + idx)
    a = _ints((m, k), 8, dt, g)
    w = _ints((n, k), 8, dt, g)
    bias = _int_bias(n, g, idx)
    code, has_res, post = _epi(epi, idx)
    res = _ints((m, n), 64, ot, g) if has_res else None
    got = _linear(a, w, bias, code, SLOPE, res, post, POST_SLOPE, ot)
    s = a.double().abs() @ w.double().abs().t() + (0 if bias is None else bias.double().abs()) + (0 if res is None else res.double().abs())
    FO.assert_exact_premise(s)
    want = FO.linear(a, w, bias, code, SLOPE, res, post, POST_SLOPE).float().to(ot)
    _assert_bits(got, want, _lin_id(case))


GROUP_SIZES = (129, 0, 1, 20000, 127, 0, 128, 2)  # 8 groups, two empty; 20000 pairs alone are 157 tiles
SEL_CASES = [(24, 16, 0, 1), (200, 20, 4, 2), (128, 264, 2, 7), (16, 512, 5, 4), (1024, 64, 1, 3), (72, 256, 3, 6)]


@pytest.mark.parametrize('case', SEL_CASES, ids=[f'k{k}-n{n}-{_NAME[IO[io][0]]}to{_NAME[IO[io][1]]}-e{e}' for k, n, io, e in SEL_CASES])
def test_linear_f16_selection_integer_exact(case):
    """out[sel_out[i]] = epilogue(A[sel_row[i]] W_g^T) for the pairs of group g; every row no pair selects keeps the exact
    bits it had (the orphans of a transposed conv rely on this)"""
    k, n, io, epi = case
    idx = SEL_CASES.index(case)
    dt, ot = IO[io]
    g = _gen(3000 + idx)
    m, n_sel = 6000, sum(GROUP_SIZES)
    n_rows = n_sel + 3001
    a = _ints((m, k), 8, dt, g)
    w = _ints((len(GROUP_SIZES) * n, k), 8, dt, g)
    sel_row = torch.randint(0, m, (n_sel,), generator=g, device='cuda', dtype=torch.int32)
    sel_out = torch.randperm(n_rows, generator=g, device='cuda')[:n_sel].to(torch.int32)
    offsets = torch.tensor(np.concatenate([[0], np.cumsum(GROUP_SIZES)]), dtype=torch.int32, device='cuda')
    rows = torch.arange(n_rows, device='cuda', dtype=F32)
    sentinel = (-(rows % 61) - 0.5)[:, None] - torch.arange(n, device='cuda', dtype=F32)[None] % 4  # exact in all three
    out = sentinel.to(ot).contiguous()
    before = out.clone()
    bias = _int_bias(n, g, idx)
    code, has_res, post = _epi(epi, idx)
    res = _ints((n_rows, n), 64, ot, g) if has_res else None
    _linear(a, w, bias, code, SLOPE, res, post, POST_SLOPE, sel=(sel_row, sel_out, offsets), out=out)
    want = FO.linear_sel(a, w, sel_row, sel_out, offsets.tolist(), before, bias, code, SLOPE, res, post, POST_SLOPE).float().to(ot)
    _assert_bits(out, want, f'selection {case}')
    untouched = torch.ones(n_rows, dtype=torch.bool, device='cuda')
    untouched[sel_out.long()] = False
    _assert_bits(out[untouched], before[untouched], 'unselected rows')


# ---- (b) error bound on random data --------------------------------------------------------------------------------------
BOUND_CONV = [(16, 16, 27, 1000, F16), (24, 17, 27, 45000, BF16), (136, 300, 32, 3000, F16), (512, 512, 32, 5000, BF16),
              (264, 100, 8, 129, F16), (64, 256, 28, 20000, BF16), (40, 255, 2, 128, F16)]
BOUND_LIN = [(3000, 2048, 264, F16), (40000, 24, 20, BF16), (129, 1024, 1024, F16), (128, 200, 512, BF16)]


def _random_inputs(shape_a, shape_w, fan_in, dt, g, big_rows):
    """random-normal inputs with `big_rows` rows scaled by 2^12 (their outputs overflow fp16), weights N(0, 1/fan_in)"""
    a = torch.randn(shape_a, generator=g, device='cuda')
    a[big_rows] *= 4096.0
    w = torch.randn(shape_w, generator=g, device='cuda') / fan_in ** 0.5
    return a.to(dt), w.to(dt)


def _random_bias(n, g):
    """N(0, 0.01) with column 0 at 1e5 and column 1 at -1e7: they overflow fp16 (+inf, and -inf after two slopes of 0.2
    and 0.1) in every row"""
    b = torch.randn(n, generator=g, device='cuda') * 0.1
    b[0], b[1] = 1e5, -1e7
    return b


def _dyadic_res(shape, g):
    """residual values exact in fp16, bf16 and fp32 (k / 16 with |k| < 128), so the three launches add the same numbers"""
    return torch.randint(-127, 128, shape, generator=g, device='cuda').to(F32) / 16


def _check_bound_and_casts(launch, ref, s, n_terms, what):
    """launch(out_dtype, residual dtype) -> output.  Asserts the fp32 result within the bound, the same launch twice
    bit-identical, and the fp16 / bf16 outputs equal to the round-to-nearest cast of the fp32 one."""
    got = launch(F32)
    err = (got.double() - ref).abs()
    b = FO.bound(s, n_terms)
    ratio = float((err / b.clamp(min=1e-300)).max())
    print(f'\n{what}: max err/bound = {ratio:.4f}  (max err {float(err.max()):.3e})')
    assert bool((err <= b).all()), f'{what}: error bound exceeded, max err/bound = {ratio}'
    _assert_bits(launch(F32), got, f'{what}: second launch')
    for ot in (F16, BF16):
        cast = got.to(ot)
        if ot == F16:
            assert bool(torch.isinf(cast).any()), 'the case must contain rows that overflow fp16'
        _assert_bits(launch(ot), cast, f'{what}: {_NAME[ot]} output')
    return ratio


@pytest.mark.parametrize('case', BOUND_CONV, ids=[f'ci{c[0]}-co{c[1]}-kv{c[2]}-n{c[3]}-{_NAME[c[4]]}' for c in BOUND_CONV])
def test_spconv_f16_error_bound_and_output_casts(case):
    ci, co, kv, n_out, dt = case
    idx = BOUND_CONV.index(case)
    g = _gen(4000 + idx)
    n_in = n_out + 17
    f, w_t = _random_inputs((n_in, ci), (kv, co, ci), kv * ci, dt, g, torch.arange(0, n_in, 97, device='cuda'))
    table = FO.build_table(FO.BUILDERS[idx % len(FO.BUILDERS)], kv, n_out, n_in, seed=idx).cuda()
    bias = _random_bias(co, g)
    res = _dyadic_res((n_out, co), g)
    slope, post_slope = float(np.float32(0.2)), float(np.float32(0.1))
    launch = lambda ot: _conv(f, w_t, table, n_out, bias, FO.ACT_LEAKY, slope, res.to(ot), FO.ACT_LEAKY, post_slope, ot)  # noqa: E731
    ref = FO.spconv(f, w_t, table, bias, FO.ACT_LEAKY, slope, res, FO.ACT_LEAKY, post_slope)
    s = FO.abs_sum(f, w_t, table, bias, res)
    _check_bound_and_casts(launch, ref, s, kv * ci, f'spconv {case}')


@pytest.mark.parametrize('case', BOUND_LIN, ids=[f'm{c[0]}-k{c[1]}-n{c[2]}-{_NAME[c[3]]}' for c in BOUND_LIN])
def test_linear_f16_error_bound_and_output_casts(case):
    m, k, n, dt = case
    g = _gen(5000 + BOUND_LIN.index(case))
    a, w = _random_inputs((m, k), (n, k), k, dt, g, torch.arange(0, m, 61, device='cuda'))
    bias = _random_bias(n, g)
    res = _dyadic_res((m, n), g)
    launch = lambda ot: _linear(a, w, bias, FO.ACT_RELU, 0.0, res.to(ot), FO.ACT_NONE, 0.0, ot)  # noqa: E731
    ref = FO.linear(a, w, bias, FO.ACT_RELU, 0.0, res)
    s = a.double().abs() @ w.double().abs().t() + bias.double().abs() + res.double().abs()
    _check_bound_and_casts(launch, ref, s, k, f'linear {case}')


# ---- (c) invariances -----------------------------------------------------------------------------------------------------
@pytest.fixture
def sm_budget():
    """sets the library's cap on the SMs of the persistent GEMM grids (a process-wide setting of the library, not of the
    device) and restores the default, all SMs, afterwards"""
    lib = _lib().load()
    yield lambda n: lib.fpcc_set_sm_budget(n)
    lib.fpcc_set_sm_budget(0)


def test_sm_budget_does_not_change_a_bit(sm_budget):
    """one CTA walking all 314 tiles flips every accumulator and metadata slot phase many times; the results of every
    budget are the bits of the full grid"""
    g = _gen(6000)
    n_out, n_in, ci, co, kv = 20000, 20100, 40, 300, 27
    f = torch.randn((n_in, ci), generator=g, device='cuda').to(BF16)
    w_t = (torch.randn((kv, co, ci), generator=g, device='cuda') / 30).to(BF16)
    table = FO.empty_tile_table(kv, n_out, n_in, 0.4, 6).cuda()
    bias = torch.randn(co, generator=g, device='cuda')
    res = torch.randn((n_out, co), generator=g, device='cuda')
    a = torch.randn((5000, 264), generator=g, device='cuda').to(F16)
    w8 = (torch.randn((8 * 48, 264), generator=g, device='cuda') / 16).to(F16)
    sizes = (300, 0, 1, 1000, 127, 0, 128, 129)
    sel_row = torch.randint(0, 5000, (sum(sizes),), generator=g, device='cuda', dtype=torch.int32)
    sel_out = torch.randperm(sum(sizes) + 100, generator=g, device='cuda')[:sum(sizes)].to(torch.int32)
    offsets = torch.tensor(np.concatenate([[0], np.cumsum(sizes)]), dtype=torch.int32, device='cuda')

    def run():
        conv = _conv(f, w_t, table, n_out, bias, FO.ACT_LEAKY, 0.2, res, FO.ACT_RELU, 0.0, F32)
        lin = _linear(a, w8[:48], None, FO.ACT_NONE, 0.0, None, FO.ACT_NONE, 0.0, F16)
        sel = _linear(a, w8, None, FO.ACT_RELU, 0.0, sel=(sel_row, sel_out, offsets),
                      out=torch.full((sum(sizes) + 100, 48), -3.0, dtype=F32, device='cuda'))
        return conv, lin, sel

    base = run()
    for budget in (1, 5, 0):
        sm_budget(budget)
        for x, y, name in zip(run(), base, ('conv', 'linear', 'selection')):
            _assert_bits(x, y, f'{name} under sm_budget({budget})')


@pytest.mark.parametrize('out_dtype', [F32, F16], ids=['f32', 'f16'])
def test_row_perm_gives_the_unpermuted_bits(out_dtype):
    """a random output-row permutation with its permuted table (not only group_rows' pattern sort) and a residual: the
    tiles hold other rows and other offset masks, but each row's sum is the same, so the bits are too"""
    g = _gen(7000)
    n_out, n_in, ci, co, kv = 30000, 25000, 24, 100, 27
    f = torch.randn((n_in, ci), generator=g, device='cuda').to(F16)
    w_t = (torch.randn((kv, co, ci), generator=g, device='cuda') / 25).to(F16)
    table = FO.random_table(kv, n_out, n_in, 0.3, 7).cuda()
    tp, perm = FO.permute_rows(table.cpu(), 8)
    bias = torch.randn(co, generator=g, device='cuda')
    res = torch.randn((n_out, co), generator=g, device='cuda').to(out_dtype)
    want = _conv(f, w_t, table, n_out, bias, FO.ACT_LEAKY, 0.2, res, FO.ACT_LEAKY, 0.1, out_dtype)
    got = _conv(f, w_t, tp.cuda(), n_out, bias, FO.ACT_LEAKY, 0.2, res, FO.ACT_LEAKY, 0.1, out_dtype, row_perm=perm.cuda())
    _assert_bits(got, want, 'row_perm')


# ---- (d) weight gradient -------------------------------------------------------------------------------------------------
WG_C_IN = (16, 24, 100, 128, 129, 200, 256)
WG_C_OUT = (1, 3, 17, 30, 40, 64, 65, 192, 256)
PAIR_COUNTS = (0, 1, 63, 64, 65, 2047, 2048, 2049, 10000)


def _pairs(counts, n_in, n_out, g):
    n = sum(counts)
    in_map = torch.randint(0, n_in, (n,), generator=g, device='cuda', dtype=torch.int32)
    out_map = torch.randint(0, n_out, (n,), generator=g, device='cuda', dtype=torch.int32)
    return in_map, out_map, [0] + np.cumsum(counts).tolist()


def _wgrad_exact(ci, co, dt, counts, seed, r=8):
    from fastpcc_b200 import ops
    g = _gen(seed)
    n_in, n_out = 3000, 2500
    x = _ints((n_in, ci), r, dt, g)
    dy = _ints((n_out, co), r, dt, g)
    in_map, out_map, off = _pairs(counts, n_in, n_out, g)
    got = ops.spconv_wgrad_f16(x, dy, in_map, out_map, off, ci, co)
    FO.assert_exact_premise(FO.wgrad(x.abs(), dy.abs(), in_map, out_map, off))
    want = FO.wgrad(x, dy, in_map, out_map, off).float()
    _assert_bits(got.reshape(-1, co), want.reshape(-1, co), f'wgrad ci{ci} co{co}')
    for k, c in enumerate(counts):
        if c == 0:
            assert bool((got[k] == 0).all()), f'offset {k} has no pairs but a nonzero gradient'
    return got


WG_CASES = [(ci, co) for ci in WG_C_IN for co in WG_C_OUT]


@pytest.mark.parametrize('ci,co', WG_CASES, ids=[f'ci{a}-co{b}' for a, b in WG_CASES])
def test_wgrad_f16_integer_exact(ci, co):
    """every pair count of PAIR_COUNTS in one call, rotated over the offsets from case to case"""
    idx = WG_CASES.index((ci, co))
    counts = PAIR_COUNTS[idx % 9:] + PAIR_COUNTS[:idx % 9]
    _wgrad_exact(ci, co, (F16, BF16)[idx % 2], counts, 8000 + idx)


def test_wgrad_f16_more_tiles_than_sms():
    _wgrad_exact(200, 65, BF16, (20000,) * 32, 8100, r=4)  # 320 tiles of 2048 pairs (and one of 1568 per offset)


def test_wgrad_f16_under_sm_budget_one(sm_budget):
    counts = (2049, 0, 65, 10000, 1, 64, 2048, 63, 0)
    full = _wgrad_exact(129, 30, F16, counts, 8200)
    sm_budget(1)
    _assert_bits(_wgrad_exact(129, 30, F16, counts, 8200), full, 'wgrad under sm_budget(1)')


def test_wgrad_f16_abi_accumulates_into_dw(sm_budget):
    """fpcc_spconv_wgrad_f16 called directly: dw is ACCUMULATED into (here: pre-filled integers); padding columns of
    x and dy hold non-zero values that must not reach dW; the tile list splits an offset at odd points and contains a tile
    of no pairs, which must leave the next tile of its CTA whole (one CTA walks them all)"""
    g = _gen(8300)
    ci, co, cip, cop, kv = 100, 30, 128, 64, 4
    n_in, n_out = 4000, 3500
    x = _ints((n_in, cip), 8, F16, g)
    dy = _ints((n_out, cop), 8, F16, g)
    counts = (3000, 0, 2049, 700)
    in_map, out_map, off = _pairs(counts, n_in, n_out, g)
    tiles = [(0, 0, 1000, 0), (0, 1000, 3000, 0), (1, 3000, 3000, 0), (2, 3000, 3001, 0), (2, 3001, 5049, 0),
             (3, 5049, 5049, 0), (3, 5049, 5749, 0)]
    tl = torch.tensor(tiles, dtype=torch.int32, device='cuda')
    dw = _ints((kv, ci, co), 100, F32, g)
    before = dw.clone()
    sm_budget(1)
    _lib().call('fpcc_spconv_wgrad_f16', _p(x), _p(dy), 0, cip, cop, _p(in_map), _p(out_map), _p(tl), len(tiles), _p(dw), ci, co,
                _stream())
    want = (before.double() + FO.wgrad(x[:, :ci], dy[:, :co], in_map, out_map, off)).float()
    _assert_bits(dw.reshape(-1, co), want.reshape(-1, co), 'wgrad accumulated into dw')
    _assert_bits(dw[1], before[1], 'offset without pairs')


# ---- (e) 64-bit offsets --------------------------------------------------------------------------------------------------
def test_spconv_f16_byte_offsets_beyond_2_31():
    """input rows at byte offsets up to 2.2e9 (8.5 M rows x 128 fp16) and fp32 output rows beyond 2^31 bytes
    (2.1 M rows x 256); sampled rows, the last tiles included, against the oracle.  About 4.4 GB of device memory."""
    g = _gen(9000)
    n_in, ci, n_out, co, kv = 8_500_000, 128, 2_100_000, 256, 2
    assert n_in * ci * 2 > 2 ** 31 and n_out * co * 4 > 2 ** 31
    f = torch.zeros((n_in, ci), dtype=F16, device='cuda')
    hi = 300_000
    f[n_in - hi:] = _ints((hi, ci), 8, F16, g)
    f[0] = _ints((1, ci), 8, F16, g)[0]
    w_t = _ints((kv, co, ci), 8, F16, g)
    table = torch.randint(n_in - hi + 1, n_in + 1, (kv, n_out), generator=g, device='cuda', dtype=torch.int32)
    table[1, ::5] = 0
    table[0, 7::11] = 1
    table[:, -1] = n_in
    bias = torch.randperm(co, generator=g, device='cuda').to(F32)
    out = _conv(f, w_t, table, n_out, bias, FO.ACT_NONE, 0.0, None, FO.ACT_NONE, 0.0, F32)
    rows = torch.cat([torch.arange(0, 256, device='cuda'), torch.arange(n_out - 384, n_out, device='cuda'),
                      torch.randint(0, n_out, (2000,), generator=g, device='cuda')])
    sub = table[:, rows]
    FO.assert_exact_premise(FO.abs_sum(f, w_t, sub, bias))
    want = FO.spconv(f, w_t, sub, bias).float()
    _assert_bits(out[rows], want, 'rows beyond 2^31 bytes')
