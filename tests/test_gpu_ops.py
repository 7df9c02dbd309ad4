"""GPU parity tests of the individual kernels against the CPU oracle, called through the C ABI
(fastpcc_b200.ops -> libfastpcc_b200.so).  Bit-exact: every comparison is array equality."""
import numpy as np
import pytest
import torch

from fastpcc_b200 import synth
from oracle import int_ops as K

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def ops():
    from fastpcc_b200 import ops as _ops
    return _ops


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _cloud(seed, n=3000, bits=7, batch=1):
    rng = np.random.default_rng(seed)
    out = []
    for b in range(batch):
        pts = np.unique(rng.integers(0, 1 << bits, (n, 3)), axis=0).astype(np.int32)
        out.append(synth.with_batch(pts, b))
    return np.concatenate(out)


@pytest.mark.parametrize('ks,st', [((3, 3, 3), (1, 1, 1)), ((2, 2, 2), (2, 2, 2)), ((4, 4, 4), (4, 4, 4))])
def test_kernel_map_lookup_and_compaction(ops, ks, st):
    C = _cloud(0, batch=2)
    if st == (1, 1, 1):
        out_c = C
    else:
        oc = C.copy(); oc[:, 1:] //= st[0]
        out_c = np.unique(oc, axis=0)
    want = K.lookup_coords(C, out_c, ks, st)
    keys, vals = ops.hash_build(dev(C))
    table = ops.kmap_lookup(keys, vals, dev(out_c), ks, st)
    assert (table.cpu().numpy() == want).all()
    # reference layout [n_pad, kvol] through the mirror class (coords permuted to x,y,z,b)
    from fastpcc_b200.int_sparse_conv import ext
    ht = ext.GPUHashTable(torch.zeros(2 * C.shape[0], dtype=torch.int64, device='cuda'),
                          torch.zeros(2 * C.shape[0], dtype=torch.int32, device='cuda'))
    ht.insert_coords(dev(C[:, [1, 2, 3, 0]]))
    t2 = ht.lookup_coords(dev(out_c[:, [1, 2, 3, 0]]), torch.tensor(ks, dtype=torch.int32, device='cuda'),
                          torch.tensor(st, dtype=torch.int32, device='cuda'), int(np.prod(ks)))
    assert t2.shape[0] % 128 == 0 and (t2[:out_c.shape[0]].T.cpu().numpy() == want).all()
    assert (t2[out_c.shape[0]:] == 0).all()
    # compaction == cuda_ops.py:132-151
    omit = 13 if ks == (3, 3, 3) else -1
    in_map, out_map, offsets = ops.kmap_compact(table, omit)
    off = offsets.cpu().numpy()
    ref = K.compact_kernel_map(want, omit)
    for k, (im, om) in enumerate(ref):
        a, b = off[k], off[k + 1]
        if im is None:
            assert a == b
        else:
            assert (in_map[a:b].cpu().numpy() == im).all() and (out_map[a:b].cpu().numpy() == om).all()


def test_downsample_upsample_roundtrip(ops):
    from oracle.lossl_coord_int import morton_xmajor
    C = _cloud(3, n=5000, bits=8, batch=2)
    order = np.lexsort((morton_xmajor(C[:, 1:]), C[:, 0]))
    C = C[order]
    # morton codes agree with the oracle
    codes = ops.morton_encode(dev(C), col0=1, msb_axis=0).cpu().numpy()
    assert (codes == morton_xmajor(C[:, 1:])).all()
    pc, occ, par, slot, cnt = ops.downsample(dev(C))
    n2 = int(cnt.item())
    oc = C.copy(); oc[:, 1:] >>= 1
    keep = np.ones(len(oc), bool); keep[1:] = (oc[1:] != oc[:-1]).any(1)
    want_c = oc[keep]
    assert n2 == want_c.shape[0] and (pc[:n2].cpu().numpy() == want_c).all()
    # occupancy bits == fold2bin conv of the reference (model.py:271-277)
    ones = np.ones((C.shape[0], 1), np.int8)
    f, _ = K.sparse_conv_in8w8out32(ones, np.eye(8, dtype=np.int8).reshape(8, 8, 1), C, want_c, (2, 2, 2), (2, 2, 2), None, None, True)
    bits = ops.occ_to_bits(occ[:n2].contiguous()).cpu().numpy()
    assert (bits == f).all()
    assert (par.cpu().numpy() == np.cumsum(keep) - 1).all()
    assert (slot.cpu().numpy() == ((C[:, 1] & 1) << 2 | (C[:, 2] & 1) << 1 | (C[:, 3] & 1))).all()
    cc, cpar, cslot, nchild = ops.upsample(pc[:n2].contiguous(), occ[:n2].contiguous())
    assert nchild == C.shape[0] and (cc.cpu().numpy() == C).all()
    assert (cpar.cpu().numpy() == par.cpu().numpy()).all() and (cslot.cpu().numpy() == slot.cpu().numpy()).all()


def test_kernel_map_from_parent_level_equals_hash_lookup(ops):
    """Octree neighbour finding (fpcc_kmap_from_parent) gives exactly the hash-built 3x3x3 table, level after level."""
    from oracle.lossl_coord_int import morton_xmajor
    C = _cloud(11, n=20000, bits=6, batch=3)
    C = C[np.lexsort((morton_xmajor(C[:, 1:]), C[:, 0]))]
    lv = [dev(C)]
    meta = []
    for _ in range(4):                                              # fine -> coarse
        pc, occ, par, slot, cnt = ops.downsample(lv[-1])
        n2 = int(cnt.item())
        meta.append((occ[:n2].contiguous(), par.contiguous(), slot.contiguous()))
        lv.append(pc[:n2].contiguous())
    keys, vals = ops.hash_build(lv[-1])
    table = ops.kmap_lookup(keys, vals, lv[-1], (3, 3, 3), (1, 1, 1))  # coarsest level: hash
    for l in range(3, -1, -1):                                      # derive every finer level from its parent level
        occ, par, slot = meta[l]
        table = ops.kmap_from_parent(table, occ, par, slot)
        keys, vals = ops.hash_build(lv[l])
        want = ops.kmap_lookup(keys, vals, lv[l], (3, 3, 3), (1, 1, 1))
        assert torch.equal(table, want), l


def _epi_args(rng, ch, prelu, out8, zp=True):
    mul = rng.integers(1 << 18, 1 << 22, ch).astype(np.uint32)
    z = np.array([int(rng.integers(-(1 << 20), 1 << 20)) if zp else 0], np.int64)
    slope = np.array([int(0.25 * (1 << 25))], np.int32) if prelu else None
    shift = 24 if out8 else 6
    return mul, z, slope, shift


@pytest.mark.parametrize('cin,cout', [(1, 16), (8, 32), (16, 16), (64, 48), (100, 30), (128, 128), (264, 64)])
@pytest.mark.parametrize('prelu,out8', [(True, True), (False, False)])
def test_fused_sparse_conv(ops, cin, cout, prelu, out8):
    rng = np.random.default_rng(cin * 1000 + cout)
    C = _cloud(5, n=2500, bits=6)
    n = C.shape[0]
    f = rng.integers(-128, 128, (n, cin)).astype(np.int8)
    w = rng.integers(-127, 128, (27, cout, cin)).astype(np.int8)
    bias = rng.integers(-5000, 5000, cout).astype(np.int32)
    mul, zp, slope, shift = _epi_args(rng, cout, prelu, out8)
    acc, _ = K.sparse_conv_in8w8out32(f, w, C, C, (3, 3, 3), (1, 1, 1), None, None, True)
    want = K.requant(acc, mul, zp, shift, np.int8 if out8 else np.int32, bias=bias, slope=slope)
    keys, vals = ops.hash_build(dev(C))
    table = ops.kmap_lookup(keys, vals, dev(C), (3, 3, 3), (1, 1, 1))
    ep = ops.make_epilogue(dev(mul), dev(zp), shift, ops.OUT_I8 if out8 else ops.OUT_I32, bias=dev(bias),
                           slope=dev(slope) if prelu else None)
    got = ops.spconv(dev(f), dev(w), table, ep)
    assert (got.cpu().numpy() == want).all()
    if ops.gemm_engine(cin, cout, 27) == 'tc':
        # rows regrouped by neighbour pattern (tile-level offset skipping): same values, original row order
        tp, perm = ops.group_rows(table)
        pn = perm.cpu().numpy()
        assert (np.sort(pn) == np.arange(n)).all() and (tp.cpu().numpy() == table.cpu().numpy()[:, pn]).all()
        masks = ((table.cpu().numpy()[:, pn] != 0).astype(np.int64) << np.arange(27)[:, None]).sum(0)
        assert (np.diff(masks) >= 0).all()
        got = ops.spconv(dev(f), dev(w), tp, ep, row_perm=perm)
        assert (got.cpu().numpy() == want).all()
    # raw accumulator + mirror API of the reference (per-offset gather-GEMM-scatter, dense centre GEMM)
    raw = ops.spconv(dev(f), dev(w), table, ops.identity_epilogue(torch.device('cuda', 0)))
    assert (raw.cpu().numpy() == acc).all()


def test_residual_epilogue_and_zero_point_comp(ops):
    rng = np.random.default_rng(9)
    C = _cloud(6, n=1500, bits=6)
    n, ch = C.shape[0], 32
    f = rng.integers(-128, 128, (n, ch)).astype(np.int8)
    w = rng.integers(-127, 128, (27, ch, ch)).astype(np.int8)
    bias = rng.integers(-5000, 5000, ch).astype(np.int32)
    comp = rng.integers(-3000, 3000, (27, ch)).astype(np.int32)
    res = rng.integers(-2 ** 31, 2 ** 31 - 1, (n, ch)).astype(np.int32)
    mul, zp, _, shift = _epi_args(rng, ch, False, False, zp=False)
    post = np.array([int(0.1 * (1 << 25))], np.int32)
    acc, _ = K.sparse_conv_in8w8out32(f, w, C, C, (3, 3, 3), (1, 1, 1), None, comp, True)
    y = K.requant(acc, mul, zp, shift, np.int32, bias=bias)
    want = K.prelu(K._wrap32(res.astype(np.int64) + y.astype(np.int64)), post)
    keys, vals = ops.hash_build(dev(C))
    table = ops.kmap_lookup(keys, vals, dev(C), (3, 3, 3), (1, 1, 1))
    ep = ops.make_epilogue(dev(mul), dev(zp), shift, ops.OUT_I32, bias=dev(bias), residual=dev(res), post_slope=dev(post))
    got = ops.spconv(dev(f), dev(w), table, ep, zp_comp=dev(comp))
    assert (got.cpu().numpy() == want).all()


@pytest.mark.parametrize('m,k,n', [(1, 16, 8), (777, 264, 255), (300, 128, 2048), (64, 7, 5), (1000, 512, 256)])
def test_linear_and_gemm(ops, m, k, n):
    rng = np.random.default_rng(m + k + n)
    a = rng.integers(-128, 128, (m, k)).astype(np.int8)
    w = rng.integers(-127, 128, (n, k)).astype(np.int8)
    bias = rng.integers(-100000, 100000, n).astype(np.int32)
    mul, zp, slope, shift = _epi_args(rng, n, True, False)
    want = K.requant(K.gemm_int8(a, w, bias), mul, zp, shift, np.int32, slope=slope)
    ep = ops.make_epilogue(dev(mul), dev(zp), shift, ops.OUT_I32, bias=dev(bias), slope=dev(slope))
    got = ops.linear(dev(a), dev(w), ep)
    assert (got.cpu().numpy() == want).all()
    from fastpcc_b200.int_sparse_conv import ext
    d = torch.empty((m, n), dtype=torch.int32, device='cuda')
    ext.cutlass_gemm_int8(dev(a), dev(w), dev(bias), d)
    assert (d.cpu().numpy() == K.gemm_int8(a, w, bias)).all()
    full = rng.integers(-1000, 1000, (m, n)).astype(np.int32)
    ext.cutlass_gemm_int8(dev(a), dev(w), dev(full), d)
    assert (d.cpu().numpy() == K.gemm_int8(a, w, full)).all()
    ext.cutlass_gemm_int8(dev(a), dev(w), torch.empty(0, dtype=torch.int32, device='cuda'), d)
    assert (d.cpu().numpy() == K.gemm_int8(a, w, None)).all()


def test_epilogue_ranges_fast_and_wide_paths(ops):
    """The tcgen05 epilogue has a 32-bit fast path guarded by range preconditions and a 64-bit general path: sweep
    shifts, multipliers up to 2^32, large biases, huge zero points, slopes outside [0, 1] and every output type so
    that both paths and the per-chunk fall-back are compared with the oracle (bias_prelu_requant.cu:6-37)."""
    rng = np.random.default_rng(7)
    m, k, n = 300, 64, 96
    a = rng.integers(-128, 128, (m, k)).astype(np.int8)
    w = rng.integers(-127, 128, (n, k)).astype(np.int8)
    acc0 = K.gemm_int8(a, w, None)
    assert ops.gemm_engine(k, n) == 'tc'
    cases = 0
    for trial in range(72):
        out_t, np_t = [(ops.OUT_I8, np.int8), (ops.OUT_I16, np.int16), (ops.OUT_I32, np.int32)][trial % 3]
        shift = int(rng.integers(0, 32))
        mul_hi = [1 << 8, 1 << 20, (1 << 31) - 1, (1 << 32) - 1][int(rng.integers(0, 4))]
        mul = rng.integers(0, mul_hi, n, endpoint=True).astype(np.uint32)
        if trial % 5 == 0:
            mul[::7] = 0
        bias_hi = [1000, 1 << 20, 1 << 29, (1 << 31) - 1][int(rng.integers(0, 4))]
        bias = rng.integers(-bias_hi, bias_hi, n, endpoint=True).astype(np.int32)
        zp = np.array([[0, 0, 1, -1, 3 << shift, -(5 << shift), (1 << 40) + 12345, -(1 << 45)][int(rng.integers(0, 8))]], np.int64)
        slope = [None, None, 0, 1 << 25, int(0.2 * (1 << 25)), -(1 << 23), 3 << 25][int(rng.integers(0, 7))]
        slope = None if slope is None else np.array([slope], np.int32)
        want = K.requant(acc0, mul, zp, shift, np_t, bias=bias, slope=slope)
        ep = ops.make_epilogue(dev(mul), dev(zp), shift, out_t, bias=dev(bias), slope=None if slope is None else dev(slope))
        got = ops.linear(dev(a), dev(w), ep).cpu().numpy()
        assert got.dtype == np_t and (got == want).all(), (trial, shift, mul_hi, bias_hi, int(zp[0]), slope)
        cases += 1
    # shifts 32..62 (the high-word fast path: the int32-producing layers and most linears of a converted model sit at
    # 36-39): same sweep, zero points on both sides of the 2^60 precondition
    for trial in range(60):
        out_t, np_t = [(ops.OUT_I8, np.int8), (ops.OUT_I16, np.int16), (ops.OUT_I32, np.int32)][trial % 3]
        shift = int(rng.integers(32, 63))
        mul_hi = [1 << 20, (1 << 30) + 12345, (1 << 31) - 1, (1 << 32) - 1][int(rng.integers(0, 4))]
        mul = rng.integers(mul_hi >> 2, mul_hi, n, endpoint=True).astype(np.uint32)
        if trial % 7 == 0:
            mul[::5] = 0
        bias_hi = [1000, 1 << 20, 1 << 29, (1 << 31) - 1][int(rng.integers(0, 4))]
        bias = rng.integers(-bias_hi, bias_hi, n, endpoint=True).astype(np.int32)
        zs = min(shift, 57)
        zp = np.array([[0, 0, 1, -1, 3 << zs, -(5 << zs), (1 << 40) + 12345, -(1 << 45), 1 << 60, -(1 << 60) - 1][int(rng.integers(0, 10))]], np.int64)
        slope = [None, None, 0, 1 << 25, int(0.2 * (1 << 25)), -(1 << 23), 3 << 25][int(rng.integers(0, 7))]
        slope = None if slope is None else np.array([slope], np.int32)
        want = K.requant(acc0, mul, zp, shift, np_t, bias=bias, slope=slope)
        ep = ops.make_epilogue(dev(mul), dev(zp), shift, out_t, bias=dev(bias), slope=None if slope is None else dev(slope))
        got = ops.linear(dev(a), dev(w), ep).cpu().numpy()
        assert got.dtype == np_t and (got == want).all(), ('hi', trial, shift, mul_hi, bias_hi, int(zp[0]), slope)
    # occupancy row bias with entries large enough to leave the proven range (per-chunk fall-back) + residual / post PReLU
    table = rng.integers(-(1 << 31), (1 << 31) - 1, (256, n), endpoint=True).astype(np.int32)
    table[:128] >>= 9
    idx = rng.integers(0, 256, m).astype(np.uint8)
    mul = rng.integers(1 << 10, 1 << 22, n).astype(np.uint32)
    bias = rng.integers(-(1 << 28), 1 << 28, n).astype(np.int32)
    for out_t, np_t, shift in [(ops.OUT_I8, np.int8, 20), (ops.OUT_I32, np.int32, 9), (ops.OUT_I8, np.int8, 38), (ops.OUT_I32, np.int32, 37)]:
        for zpv in (0, 77777):
            zp = np.array([zpv], np.int64)
            slope = np.array([int(0.3 * (1 << 25))], np.int32)
            accb = (acc0.astype(np.int64) + table[idx].astype(np.int64)).astype(np.int32)  # int32 add wraps
            want = K.requant(accb, mul, zp, shift, np_t, bias=bias, slope=slope)
            ep = ops.make_epilogue(dev(mul), dev(zp), shift, out_t, bias=dev(bias), slope=dev(slope), row_bias=(dev(table), dev(idx)))
            got = ops.linear(dev(a), dev(w), ep).cpu().numpy()
            assert (got == want).all(), (out_t, zpv)
    res = rng.integers(-(1 << 31), (1 << 31) - 1, (m, n), endpoint=True).astype(np.int32)
    for post_v in (int(0.25 * (1 << 25)), -(1 << 24), 5 << 25):
        post = np.array([post_v], np.int32)
        zp = np.zeros(1, np.int64)
        y = K.requant(acc0, mul, zp, 3, np.int32, bias=bias)
        want = K.prelu((y.astype(np.int64) + res.astype(np.int64)).astype(np.int32), post)
        ep = ops.make_epilogue(dev(mul), dev(zp), 3, ops.OUT_I32, bias=dev(bias), residual=dev(res), post_slope=dev(post))
        got = ops.linear(dev(a), dev(w), ep).cpu().numpy()
        assert (got == want).all(), post_v
    assert cases == 72
    # stand-alone requant with one multiplier (RequantFxpToScaledInt8, cuda_ops.py:478-507): full int32 inputs
    x = rng.integers(-(1 << 31), (1 << 31) - 1, (513, 64), endpoint=True).astype(np.int32)
    x[0, :8] = [-(1 << 31), (1 << 31) - 1, 0, -1, 1, -(1 << 31) + 1, 1 << 30, -(1 << 30)]
    for shift in (0, 1, 7, 23, 31, 32, 36, 48, 62):
        for mulv in (0, 1, 3, 12345, (1 << 22) + 5, (1 << 30) + 99, (1 << 31) - 1, (1 << 31) + 7):
            for zpv in (0, -1, 5 << min(shift, 57), -(1 << 40), (1 << 60) - 1, -(3 << 58)):
                mul1, zp = np.array([mulv], np.uint32), np.array([zpv], np.int64)
                want = K.requant(x, np.full(64, mulv, np.uint32), zp, shift, np.int8)
                got = ops.requant(dev(x), ops.make_epilogue(dev(mul1), dev(zp), shift, ops.OUT_I8)).cpu().numpy()
                assert (got == want).all(), (shift, mulv, zpv)
    # ... and with the PReLU in front (prelu_requant_to_int8, bias_prelu_requant.cu:6-37): slopes inside and outside [0, 1]
    for slope_v in (0, 1 << 25, int(0.3 * (1 << 25)), -(1 << 22), 3 << 25):
        for shift, mulv, zpv in ((7, 12345, 0), (23, (1 << 22) + 5, -77), (31, 3, 5 << 31), (36, (1 << 31) + 7, 0),
                                 (32, 3, -(5 << 33)), (48, (1 << 30) + 12345, 1 << 47), (48, (1 << 30) - 7, -(1 << 52) - 3), (62, (1 << 29) + 3, 0)):
            mul1, zp, sl = np.array([mulv], np.uint32), np.array([zpv], np.int64), np.array([slope_v], np.int32)
            want = K.requant(x, np.full(64, mulv, np.uint32), zp, shift, np.int8, slope=sl)
            got = ops.requant(dev(x), ops.make_epilogue(dev(mul1), dev(zp), shift, ops.OUT_I8, slope=dev(sl))).cpu().numpy()
            assert (got == want).all(), (slope_v, shift, mulv, zpv)


def test_epilogue_shift0_and_small_negatives(ops):
    """Shift 0 has no rounding correction (requant.cu:16-20) and must never take the 32-bit paths, whose addend folds
    the "-1 for negatives": non-zero zero points on NON-saturating negatives, through the fused linear epilogue
    (a zero accumulator whose bias carries the values) and through the stand-alone requant.  Kept as its own test so
    that it also runs first in a fresh process (round-1 open question: a one-off failure of these cases run alone)."""
    rng = np.random.default_rng(7)
    m, k, n = 300, 64, 96
    a = rng.integers(-128, 128, (m, k)).astype(np.int8)
    w = rng.integers(-127, 128, (n, k)).astype(np.int8)
    acc0 = K.gemm_int8(a, w, None)
    small = (acc0 >> 12).astype(np.int32)  # |values| < 128: inside int8
    a_s, w_s = np.zeros((m, k), np.int8), np.zeros((n, k), np.int8)
    for out_t, np_t in ((ops.OUT_I8, np.int8), (ops.OUT_I16, np.int16), (ops.OUT_I32, np.int32)):
        for shift in (0, 1, 7):
            for zpv in (0, 1, -1, 5, -(3 << shift)):
                for mulv in (1, 3):
                    mul1, zp = np.full(n, mulv, np.uint32), np.array([zpv], np.int64)
                    bias_s = small[zpv % m].copy()
                    want = K.requant(np.zeros((m, n), np.int32), mul1, zp, shift, np_t, bias=bias_s)
                    got = ops.linear(dev(a_s), dev(w_s), ops.make_epilogue(dev(mul1), dev(zp), shift, out_t, bias=dev(bias_s))).cpu().numpy()
                    assert (got == want).all(), ('bias only', out_t, shift, zpv, mulv)
                    # the same values arriving through the accumulator: small = acc0 >> 12 is not a GEMM result, so
                    # use the real accumulator with a multiplier / shift pair that keeps it unsaturated
                    want = K.requant(acc0, mul1, zp, shift + 12, np_t)
                    got = ops.linear(dev(a), dev(w), ops.make_epilogue(dev(mul1), dev(zp), shift + 12, out_t)).cpu().numpy()
                    assert (got == want).all(), ('acc', out_t, shift, zpv, mulv)
    x = rng.integers(-300, 300, (513, 64)).astype(np.int32)
    x[1, :8] = [-10, -3, -2, -7, -100, 9, -41, -127]
    x[2, :4] = [(1 << 31) - 1, -(1 << 31), (1 << 31) - 2, 0]
    for shift in (0, 1, 7, 33, 40):
        for mulv in (0, 1, 3, 77):
            for zpv in (0, 1, -1, 5, -(3 << shift), -(1 << 35)):
                mul1, zp = np.array([mulv], np.uint32), np.array([zpv], np.int64)
                want = K.requant(x, np.full(64, mulv, np.uint32), zp, shift, np.int8)
                got = ops.requant(dev(x), ops.make_epilogue(dev(mul1), dev(zp), shift, ops.OUT_I8)).cpu().numpy()
                assert (got == want).all(), ('requant', shift, mulv, zpv)


def test_requant_into_column_slices_of_one_buffer(ops):
    """fpcc_requant_ld: the two RequantFxpToScaledInt8 in front of Linear(cat(F, embed)) (lossl_coord_int/model.py:199-201)
    write the column halves of one [rows, 2C] int8 buffer; equal to requant + torch.cat, neighbours untouched."""
    rng = np.random.default_rng(3)
    rows, c1, c2 = 1237, 64, 32
    x1 = rng.integers(-(1 << 31), (1 << 31) - 1, (rows, c1), endpoint=True).astype(np.int32)
    x2 = rng.integers(-(1 << 26), 1 << 26, (rows, c2)).astype(np.int32)
    for shift, mulv, zpv, slope_v in ((48, (1 << 30) + 12345, 0, None), (40, 12345, -(3 << 39), int(0.3 * (1 << 25))), (7, 77, 5, None)):
        mul1, zp = np.array([mulv], np.uint32), np.array([zpv], np.int64)
        sl = None if slope_v is None else np.array([slope_v], np.int32)
        ep = ops.make_epilogue(dev(mul1), dev(zp), shift, ops.OUT_I8, slope=None if sl is None else dev(sl))
        buf = torch.full((rows, c1 + c2 + 16), 99, dtype=torch.int8, device='cuda')
        ops.requant(dev(x1), ep, out=buf[:, :c1])
        ops.requant(dev(x2), ep, out=buf[:, c1:c1 + c2])
        want = np.concatenate([K.requant(x1, np.full(c1, mulv, np.uint32), zp, shift, np.int8, slope=sl),
                               K.requant(x2, np.full(c2, mulv, np.uint32), zp, shift, np.int8, slope=sl)], 1)
        got = buf.cpu().numpy()
        assert (got[:, :c1 + c2] == want).all() and (got[:, c1 + c2:] == 99).all(), (shift, mulv, zpv)
    with pytest.raises(RuntimeError):
        ops.requant(dev(x1[:, :24]), ep, out=buf[:, :24])  # 24 channels: not a multiple of 16


def _tie_values(mul, zp, shift, lo, hi):
    """all v in [lo, hi] for which v*mul + zp is an exact rounding tie of `shift` (brute force, python ints)"""
    M, half = 1 << shift, 1 << (shift - 1)
    return [v for v in range(lo, hi + 1) if (v * int(mul) + int(zp)) % M == half]


@pytest.mark.parametrize('shift,tz,n', [(38, 28, 96), (30, 20, 96), (38, 28, 512), (33, 24, 96)])
def test_epilogue_tie_free_and_tie_chunks(ops, shift, tz, n):
    """int8 outputs round exact ties half away from zero on the sign-exact lean path, in 16-channel chunks with and
    without a channel that can tie inside the accumulator bound (tie analysis: csrc/epi_nt.cuh).
    Multipliers with `tz` trailing zeros make ties reachable every 2^(shift - tz) values; the occupancy row-bias table
    injects the exact tie values (negative and positive, also behind the PReLU) into a zero accumulator.  Chunk 0 has
    no tie-able channel, chunk 1 mixes one tie-able channel in, chunk 2 is all tie-able; n = 512 restages the constants
    per channel block.  Reference arithmetic: requant.cu:16-20, bias_prelu_requant.cu:6-37."""
    rng = np.random.default_rng(shift * 100 + n)
    m, k = 300, 64
    a = np.zeros((m, k), np.int8)
    w = np.zeros((n, k), np.int8)
    bound = 1 << 13
    for zpv in (0, 5 << tz, -(7 << tz) + 3):
        mul = (rng.integers(1 << 20, 1 << 30, n) | 1).astype(np.uint32)  # odd: tie-free inside the bound for these shifts
        tie_ch = [17] + list(range(32, 48)) + ([300, 511] if n > 300 else [])
        for c in tie_ch:
            mul[c] = np.uint32((2 * int(rng.integers(1, 4)) + 1) << tz)
        bias = rng.integers(-500, 500, n).astype(np.int32)
        zp = np.array([zpv], np.int64)
        for slope_v in (None, 1 << 23):  # PReLU slope 0.25: prelu(4 v) == v exactly for v < 0
            table = rng.integers(-bound + 600, bound - 600, (256, n)).astype(np.int32)
            hits = 0
            for c in tie_ch:
                ties = _tie_values(mul[c], zpv, shift, -1500, 1500)
                if zpv % (1 << tz) == 0:
                    assert ties, (c, int(mul[c]))
                for i, v in enumerate(ties[:40]):
                    tv = 4 * v if (slope_v is not None and v < 0) else v
                    table[3 + 5 * i, c] = tv - int(bias[c])
                    hits += 1
            idx = rng.integers(0, 256, m).astype(np.uint8)
            idx[:256] = np.arange(256)
            slope = None if slope_v is None else np.array([slope_v], np.int32)
            accb = table[idx].astype(np.int32)
            want = K.requant(accb, mul, zp, shift, np.int8, bias=bias, slope=slope)
            # the ties must matter: dropping the "- [r < 0]" term changes at least one output
            if hits and zpv % (1 << tz) == 0:
                v = accb.astype(np.int64) + bias.astype(np.int64)
                if slope is not None:
                    v = K.prelu(v.astype(np.int32), slope).astype(np.int64)
                naive = np.clip((v * mul.astype(np.int64) + zpv + (1 << (shift - 1))) >> shift, -128, 127)
                assert (naive != want).any()
            ep = ops.make_epilogue(dev(mul), dev(zp), shift, ops.OUT_I8, bias=dev(bias), slope=None if slope is None else dev(slope),
                                   row_bias=(dev(table), dev(idx), bound))
            got = ops.linear(dev(a), dev(w), ep).cpu().numpy()
            assert (got == want).all(), (zpv, slope_v, np.argwhere(got != want)[:5])
    # the same through the conv kernel (MODE 0: static constants, 12 epilogue warps): zero features, the bias carries
    # one value per channel -- the tie itself for the tie-able channels
    if n <= 256:
        C = _cloud(11, n=1500, bits=6)
        keys, vals = ops.hash_build(dev(C))
        tab = ops.kmap_lookup(keys, vals, dev(C), (3, 3, 3), (1, 1, 1))
        f = np.zeros((C.shape[0], 32), np.int8)
        w3 = np.zeros((27, n, 32), np.int8)
        for zpv in (0, 5 << tz):
            mul = (rng.integers(1 << 20, 1 << 30, n) | 1).astype(np.uint32)
            bias = rng.integers(-3000, 3000, n).astype(np.int32)
            for c in [17] + list(range(32, 48)):
                mul[c] = np.uint32(3 << tz)
                ties = [v for v in _tie_values(mul[c], zpv, shift, -3000, 3000) if v < 0]
                if ties:
                    bias[c] = ties[c % len(ties)]
            zp = np.array([zpv], np.int64)
            want = K.requant(np.zeros((C.shape[0], n), np.int32), mul, zp, shift, np.int8, bias=bias)
            got = ops.spconv(dev(f), dev(w3), tab, ops.make_epilogue(dev(mul), dev(zp), shift, ops.OUT_I8, bias=dev(bias))).cpu().numpy()
            assert (got == want).all(), ('conv', zpv)


@pytest.mark.parametrize('k,n', [(64, 64), (256, 256), (32, 48)])
def test_fused_second_stage_equals_prelu_then_requant(ops, k, n):
    """fpcc_epilogue::post_requant_mul: an int32 (Q8.23) linear whose only consumer is [PReLUIn32Out32 +]
    RequantFxpToScaledInt8 emits that consumer's int8 directly.  Must equal the three stand-alone steps of the
    reference (bias_requant_to_int32 -> prelu -> requant_to_int8) for plain and selection linears, symmetric and
    asymmetric second stages, values that saturate the int32 first stage (exact per-column redo) and first-stage
    parameters outside the lean path (generic epilogue)."""
    rng = np.random.default_rng(k * 1000 + n)
    m = 700
    a = rng.integers(-128, 128, (m, k)).astype(np.int8)
    w = rng.integers(-127, 128, (n, k)).astype(np.int8)
    acc = K.gemm_int8(a, w, None)
    cases = 0
    for shift1, mul_hi, bias_hi in ((9, 1 << 20, 1 << 16), (12, 1 << 22, 1 << 20), (3, 1 << 27, 1 << 28), (5, (1 << 32) - 1, 1000), (0, 7, 100)):
        mul1 = rng.integers(mul_hi >> 2, mul_hi, n, endpoint=True).astype(np.uint32)
        bias = rng.integers(-bias_hi, bias_hi, n, endpoint=True).astype(np.int32)
        zp1 = np.zeros(1, np.int64)
        y = K.requant(acc, mul1, zp1, shift1, np.int32, bias=bias)
        for shift2, mul2v, zp2v, slope2v in ((48, (1 << 30) + 12345, 0, None), (48, (1 << 29) + 7, 0, int(0.25 * (1 << 25))),
                                            (44, (1 << 30) - 3, (5 << 44) + 99, int(0.1 * (1 << 25))), (40, 12345, -(3 << 39), None),
                                            (33, (1 << 31) - 1, 1, 1 << 25), (62, (1 << 30) + 1, -(1 << 59), 0)):
            mul2, zp2 = np.array([mul2v], np.uint32), np.array([zp2v], np.int64)
            sl2 = None if slope2v is None else np.array([slope2v], np.int32)
            y2 = y if sl2 is None else K.prelu(y, sl2)
            want = K.requant(y2, np.full(n, mul2v, np.uint32), zp2, shift2, np.int8)
            post = (dev(mul2), dev(zp2), shift2, None if sl2 is None else dev(sl2))
            ep = ops.make_epilogue(dev(mul1), dev(zp1), shift1, ops.OUT_I32, bias=dev(bias), post_requant=post)
            got = ops.linear(dev(a), dev(w), ep)
            assert got.dtype == torch.int8 and (got.cpu().numpy() == want).all(), (shift1, shift2, mul2v, zp2v, slope2v)
            cases += 1
    assert cases == 30
    # selection form (Linear(C -> 8C)[child mask] of the multi-step predictors), per-group bias / multipliers
    if n % 16 == 0:
        occ = rng.integers(1, 256, m).astype(np.uint8)
        w8 = rng.integers(-127, 128, (8 * n, k)).astype(np.int8)
        bias8 = rng.integers(-100000, 100000, 8 * n).astype(np.int32)
        mul8 = rng.integers(1 << 18, 1 << 21, 8 * n).astype(np.uint32)
        dense = K.requant(K.gemm_int8(a, w8, bias8), mul8, np.zeros(1, np.int64), 10, np.int32)
        bits = ((occ[:, None] >> np.arange(7, -1, -1)[None]) & 1).astype(bool)
        y = dense.reshape(m, 8, n)[bits]
        sl2, mul2, zp2 = np.array([int(0.3 * (1 << 25))], np.int32), np.array([(1 << 30) + 77], np.uint32), np.array([3 << 45], np.int64)
        want = K.requant(K.prelu(y, sl2), np.full(n, mul2[0], np.uint32), zp2, 47, np.int8)
        C4 = np.zeros((m, 4), np.int32); C4[:, 1] = np.arange(m)
        _, par, slot, n_child = ops.upsample(dev(C4), dev(occ))
        sel = ops.slot_pairs(par, slot)
        ep = ops.make_epilogue(dev(mul8), dev(np.zeros(1, np.int64)), 10, ops.OUT_I32, bias=dev(bias8),
                               post_requant=(dev(mul2), dev(zp2), 47, dev(sl2)))
        got = ops.linear(dev(a), dev(w8), ep, sel=sel, n_out_rows=n_child)
        assert got.dtype == torch.int8 and (got.cpu().numpy() == want).all()


@pytest.mark.parametrize('k,n', [(64, 64), (256, 256)])
def test_dual_output_int32_and_fused_int8(ops, k, n):
    """fpcc_epilogue::aux_out: the int32 (Q8.23) rows AND the int8 rows of one consumer's [PReLU +] requant leave the same
    kernel.  Both must equal the stand-alone steps of the reference (bias_requant_to_int32 [+ residual + prelu], then
    prelu + requant_to_int8), for the linear (plain, PReLU, occupancy row bias), for the ResBlock conv2 form (residual +
    post PReLU, rows grouped), with first stages that saturate int32 (exact redo) and parameters outside the lean path."""
    rng = np.random.default_rng(k * 77 + n)
    m = 900
    a = rng.integers(-128, 128, (m, k)).astype(np.int8)
    w = rng.integers(-127, 128, (n, k)).astype(np.int8)
    acc = K.gemm_int8(a, w, None)
    zp1 = np.zeros(1, np.int64)
    for shift1, mul_hi, bias_hi, slope1 in ((9, 1 << 20, 1 << 16, None), (12, 1 << 22, 1 << 20, int(0.25 * (1 << 25))), (3, 1 << 27, 1 << 28, None),
                                            (5, (1 << 32) - 1, 1000, None)):
        mul1 = rng.integers(mul_hi >> 2, mul_hi, n, endpoint=True).astype(np.uint32)
        bias = rng.integers(-bias_hi, bias_hi, n, endpoint=True).astype(np.int32)
        sl1 = None if slope1 is None else np.array([slope1], np.int32)
        y = K.requant(acc, mul1, zp1, shift1, np.int32, bias=bias, slope=sl1)
        for shift2, mul2v, zp2v, slope2v in ((48, (1 << 30) + 12345, 0, None), (44, (1 << 30) - 3, (5 << 44) + 99, int(0.1 * (1 << 25))),
                                            (40, 12345, -(3 << 39), None), (62, (1 << 30) + 1, -(1 << 59), 0)):
            mul2, zp2 = np.array([mul2v], np.uint32), np.array([zp2v], np.int64)
            sl2 = None if slope2v is None else np.array([slope2v], np.int32)
            want8 = K.requant(y if sl2 is None else K.prelu(y, sl2), np.full(n, mul2v, np.uint32), zp2, shift2, np.int8)
            aux = torch.full((m, n), 77, dtype=torch.int8, device='cuda')
            ep = ops.make_epilogue(dev(mul1), dev(zp1), shift1, ops.OUT_I32, bias=dev(bias), slope=None if sl1 is None else dev(sl1),
                                   post_requant=(dev(mul2), dev(zp2), shift2, None if sl2 is None else dev(sl2)), aux_out=aux)
            got = ops.linear(dev(a), dev(w), ep)
            assert got.dtype == torch.int32 and (got.cpu().numpy() == y).all(), ('i32', shift1, shift2)
            assert (aux.cpu().numpy() == want8).all(), ('i8', shift1, shift2, mul2v, zp2v, slope2v)
    # occupancy row bias + dual output (LinearIn8W8.forward_with_bits as dec[1])
    table = rng.integers(-(1 << 20), 1 << 20, (256, n)).astype(np.int32)
    idx = rng.integers(0, 256, m).astype(np.uint8)
    mul1 = rng.integers(1 << 16, 1 << 19, n).astype(np.uint32)
    bias = rng.integers(-100000, 100000, n).astype(np.int32)
    sl1 = np.array([int(0.3 * (1 << 25))], np.int32)
    accb = (acc.astype(np.int64) + table[idx].astype(np.int64)).astype(np.int32)
    y = K.requant(accb, mul1, zp1, 8, np.int32, bias=bias, slope=sl1)
    mul2, zp2 = np.array([(1 << 30) + 5], np.uint32), np.array([3 << 44], np.int64)
    want8 = K.requant(y, np.full(n, mul2[0], np.uint32), zp2, 47, np.int8)
    aux = torch.empty((m, n), dtype=torch.int8, device='cuda')
    ep = ops.make_epilogue(dev(mul1), dev(zp1), 8, ops.OUT_I32, bias=dev(bias), slope=dev(sl1), row_bias=(dev(table), dev(idx), 1 << 20),
                           post_requant=(dev(mul2), dev(zp2), 47, None), aux_out=aux)
    got = ops.linear(dev(a), dev(w), ep)
    assert (got.cpu().numpy() == y).all() and (aux.cpu().numpy() == want8).all()
    # ResBlock conv2 form: conv + residual + post PReLU -> int32 block output, plus the next Requant's int8 rows
    if k % 16 == 0 and ops.gemm_engine(k, n, 27) == 'tc':
        C = _cloud(9, n=2000, bits=6)
        nn_ = C.shape[0]
        f = rng.integers(-128, 128, (nn_, k)).astype(np.int8)
        w3 = rng.integers(-127, 128, (27, n, k)).astype(np.int8)
        res = rng.integers(-(1 << 28), 1 << 28, (nn_, n)).astype(np.int32)
        post = np.array([int(0.2 * (1 << 25))], np.int32)
        acc3, _ = K.sparse_conv_in8w8out32(f, w3, C, C, (3, 3, 3), (1, 1, 1), None, None, True)
        y = K.prelu((K.requant(acc3, mul1, zp1, 12, np.int32, bias=bias).astype(np.int64) + res.astype(np.int64)).astype(np.int32), post)
        want8 = K.requant(y, np.full(n, mul2[0], np.uint32), zp2, 47, np.int8)
        keys, vals = ops.hash_build(dev(C))
        tb = ops.kmap_lookup(keys, vals, dev(C), (3, 3, 3), (1, 1, 1))
        tp, perm = ops.group_rows(tb)
        aux = torch.empty((nn_, n), dtype=torch.int8, device='cuda')
        ep = ops.make_epilogue(dev(mul1), dev(zp1), 12, ops.OUT_I32, bias=dev(bias), residual=dev(res), post_slope=dev(post),
                               post_requant=(dev(mul2), dev(zp2), 47, None), aux_out=aux)
        got = ops.spconv(dev(f), dev(w3), tp, ep, row_perm=perm)
        assert (got.cpu().numpy() == y).all() and (aux.cpu().numpy() == want8).all()


def test_linear_over_in_memory_concat_of_features_and_occupancy_bits(ops):
    """Linear(cat(F, bits)) (lossl_coord_int/model.py:63-64) as ONE GEMM with K = C + 16: the requant writes the first C
    columns of the buffer (fpcc_requant_ld), fpcc_occ_bits_q8 the 8 bit channels + 8 zero columns; a producer with a fused
    second stage writes its int8 rows there through fpcc_epilogue::out_ld.  Equal to the GEMM over the explicit
    concatenation and to the occupancy row-bias form."""
    rng = np.random.default_rng(21)
    m, c, n = 777, 64, 96
    x32 = rng.integers(-(1 << 27), 1 << 27, (m, c)).astype(np.int32)
    occ = rng.integers(1, 256, m).astype(np.uint8)
    q0, q1 = -7, 93
    mulr, zpr = np.array([(1 << 30) + 321], np.uint32), np.array([5 << 40], np.int64)
    f8 = K.requant(x32, np.full(c, mulr[0], np.uint32), zpr, 47, np.int8)
    bits = ((occ[:, None] >> np.arange(7, -1, -1)[None]) & 1).astype(bool)
    a_cat = np.concatenate([f8, np.where(bits, q1, q0).astype(np.int8)], 1)
    w = rng.integers(-127, 128, (n, c + 8)).astype(np.int8)
    bias = rng.integers(-50000, 50000, n).astype(np.int32)
    mul = rng.integers(1 << 20, 1 << 23, n).astype(np.uint32)
    zp = np.array([-3], np.int64)
    slope = np.array([int(0.2 * (1 << 25))], np.int32)
    want = K.requant(K.gemm_int8(a_cat, w, None), mul, zp, 30, np.int8, bias=bias, slope=slope)
    buf = torch.full((m, c + 16), 55, dtype=torch.int8, device='cuda')
    ops.requant(dev(x32), ops.make_epilogue(dev(mulr), dev(zpr), 47, ops.OUT_I8), out=buf[:, :c])
    ops.occ_bits_q8(dev(occ), q0, q1, buf[:, c:])
    assert (buf.cpu().numpy()[:, :c + 8] == a_cat).all() and (buf.cpu().numpy()[:, c + 8:] == 0).all()
    w_cat = np.concatenate([w, np.zeros((n, 8), np.int8)], 1)
    ep = ops.make_epilogue(dev(mul), dev(zp), 30, ops.OUT_I8, bias=dev(bias), slope=dev(slope))
    got = ops.linear(buf, dev(w_cat), ep).cpu().numpy()
    assert (got == want).all()
    # a producer with a fused second stage writes its int8 rows into the column slice (output pitch)
    k2 = 64
    a2 = rng.integers(-128, 128, (m, k2)).astype(np.int8)
    w2 = rng.integers(-127, 128, (c, k2)).astype(np.int8)
    mul1 = rng.integers(1 << 18, 1 << 21, c).astype(np.uint32)
    y = K.requant(K.gemm_int8(a2, w2, None), mul1, np.zeros(1, np.int64), 10, np.int32)
    want8 = K.requant(y, np.full(c, mulr[0], np.uint32), zpr, 47, np.int8)
    buf2 = torch.full((m, c + 16), 55, dtype=torch.int8, device='cuda')
    ep2 = ops.make_epilogue(dev(mul1), dev(np.zeros(1, np.int64)), 10, ops.OUT_I32, post_requant=(dev(mulr), dev(zpr), 47, None))
    ret = ops.linear(dev(a2), dev(w2), ep2, out=buf2[:, :c])
    assert ret.data_ptr() == buf2.data_ptr()
    b2 = buf2.cpu().numpy()
    assert (b2[:, :c] == want8).all() and (b2[:, c:] == 55).all()


def test_selected_linear_equals_masked_dense(ops):
    """Linear(C->8C) + child mask (model.py:64-66) == occupied-children-only evaluation."""
    rng = np.random.default_rng(4)
    n, ch = 900, 32
    a = rng.integers(-128, 128, (n, ch)).astype(np.int8)
    w = rng.integers(-127, 128, (8 * ch, ch)).astype(np.int8)
    bias = rng.integers(-100000, 100000, 8 * ch).astype(np.int32)
    mul, zp, _, shift = _epi_args(rng, 8 * ch, False, False)
    occ = rng.integers(1, 256, n).astype(np.uint8)
    dense = K.requant(K.gemm_int8(a, w, bias), mul, zp, shift, np.int32)
    bits = ((occ[:, None] >> np.arange(7, -1, -1)[None]) & 1).astype(bool)
    want = dense.reshape(n, 8, ch)[bits]
    coords = dev(synth.with_batch(np.stack([np.arange(n), np.zeros(n), np.zeros(n)], 1).astype(np.int32)))
    _, par, slot, nchild = ops.upsample(coords, dev(occ), want_coords=False)
    sel = ops.slot_pairs(par, slot)
    ep = ops.make_epilogue(dev(mul), dev(zp), shift, ops.OUT_I32, bias=dev(bias))
    got = ops.linear(dev(a), dev(w), ep, sel=sel, n_out_rows=nchild)
    assert got.shape == want.shape and (got.cpu().numpy() == want).all()


def test_mirror_gather_gemm_scatter_and_requant_family(ops):
    from fastpcc_b200.int_sparse_conv import ext
    rng = np.random.default_rng(8)
    m, k, n, L = 500, 24, 40, 320
    a = rng.integers(-128, 128, (m, k)).astype(np.int8)
    w = rng.integers(-127, 128, (n, k)).astype(np.int8)
    d0 = rng.integers(-10 ** 6, 10 ** 6, (600, n)).astype(np.int32)
    g = rng.integers(0, m, L).astype(np.int32)
    s = rng.permutation(600)[:L].astype(np.int32)
    want = d0.copy()
    K.gather_gemm_scatter_int8(a, w, want, g, s)
    d = dev(d0)
    ext.cutlass_gather_gemm_scatter_int8(dev(a), dev(w), d, d, dev(g), dev(s))
    assert (d.cpu().numpy() == want).all()
    x = rng.integers(-2 ** 31, 2 ** 31 - 1, (257, 33)).astype(np.int32)
    bias = rng.integers(-2 ** 20, 2 ** 20, 33).astype(np.int32)
    mul = rng.integers(1, 2 ** 32 - 1, 33).astype(np.uint32)
    zp = np.array([-12345678901], np.int64)
    slope = np.array([-(1 << 24)], np.int32)
    for shift in (0, 1, 17, 40):
        for name, dt in (('int8', np.int8), ('int16', np.int16), ('int32', np.int32)):
            for kind in ('', 'bias_', 'prelu_', 'bias_prelu_'):
                fn = getattr(ext, f'{kind}requant_to_{name}')
                args = [dev(x)] + ([dev(bias)] if 'bias' in kind else []) + ([dev(slope)] if 'prelu' in kind else []) \
                    + [dev(mul), dev(zp), shift]
                got = fn(*args).cpu().numpy()
                want = K.requant(x, mul, zp, shift, dt, bias=bias if 'bias' in kind else None,
                                 slope=slope if 'prelu' in kind else None)
                assert got.dtype == dt and (got == want).all(), (kind, name, shift)
    assert (ext.prelu(dev(x), dev(slope)).cpu().numpy() == K.prelu(x, slope)).all()
    with pytest.raises(RuntimeError):
        ext.requant_to_int8(dev(x), dev(mul), dev(zp), -1)


@pytest.mark.parametrize('S', [255, 2, 64, 300])
def test_softmax_and_cdf_head(ops, S):
    from fastpcc_b200.int_sparse_conv import ext
    rng = np.random.default_rng(S)
    n = 1000
    logits = (rng.normal(0, 4, (n, S)) * (1 << 23)).clip(-2 ** 31, 2 ** 31 - 1).astype(np.int32)
    logits[0] = 0
    logits[1] = -2 ** 31
    logits[2, 0] = 2 ** 31 - 1
    sm = ext.softmax_int32(dev(logits >> 7)).cpu().numpy()
    assert (sm.view(np.uint32) == K.softmax_int32(logits >> 7)).all()
    want = K.batch_quantize_pmf(logits)
    cdf = ops.quantize_cdf(dev(logits), ld=max(256, S)).cpu().numpy().view(np.uint16)
    assert (cdf[:, :S] == want).all() and (cdf[:, S:] == 0xFFFF).all()
    sym = rng.integers(0, S, n).astype(np.int32)
    sym[:3] = [0, S - 1, S - 1]
    rngs = ops.cdf_symbol_ranges(dev(logits), dev(sym)).cpu().numpy().view(np.uint32)
    w64 = want.astype(np.int64)
    lo = np.where(sym == 0, 0, w64[np.arange(n), np.maximum(sym - 1, 0)])
    hi = np.where(sym == S - 1, 65536, w64[np.arange(n), sym])
    assert ((rngs & 0xFFFF) == lo).all() and ((rngs >> 16) + 1 == hi - lo).all()
    # the same rows as a column slice of a wider (padded) buffer: the kernels take the row pitch
    pitch = (S + 15) // 16 * 16 + 16
    wide = torch.full((n, pitch), 12345, dtype=torch.int32, device='cuda')
    wide[:, :S] = dev(logits)
    cdf2 = ops.quantize_cdf(wide[:, :S], ld=max(256, S)).cpu().numpy().view(np.uint16)
    assert (cdf2 == cdf).all()
    assert (ops.cdf_symbol_ranges(wide[:, :S], dev(sym)).cpu().numpy().view(np.uint32) == rngs).all()
