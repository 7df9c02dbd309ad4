"""fp16 / bf16 tensor-core sparse convolution and linear (tcgen05.mma.kind::f16) against a plain fp32 reference of
the same op.  Tolerance (stated by BASELINE.json north_star): 1e-2 relative in fp16; bf16 has 3 fewer mantissa bits
so its bound is 4e-2.  'Relative' = max |got - want| / max |want| over the tensor."""
import numpy as np
import pytest
import torch

from fastpcc_b200 import synth
from oracle import float_ops as FO

pytestmark = pytest.mark.gpu
TOL = {torch.float16: 1e-2, torch.bfloat16: 4e-2}


def _rel(got, want):
    return float(np.abs(got.astype(np.float64) - want).max() / max(np.abs(want).max(), 1e-12))


def _cloud(seed, n, bits, stride=1):
    rng = np.random.default_rng(seed)
    pts = np.unique(rng.integers(0, 1 << bits, (n, 3)), axis=0).astype(np.int32) * stride
    return synth.with_batch(pts)


@pytest.mark.parametrize('dtype', [torch.float16, torch.bfloat16])
@pytest.mark.parametrize('cin,cout,ks', [(16, 16, 3), (64, 128, 3), (128, 128, 3), (32, 64, 2), (128, 1, 3)])
def test_spconv_f16_matches_fp32_reference(dtype, cin, cout, ks):
    from fastpcc_b200 import ops
    if cout < 16:
        pytest.skip('C_out < 16 runs through the padded path of the layer API (tested there)')
    rng = np.random.default_rng(cin + cout)
    ts = 2
    C = _cloud(1, 4000, 6, stride=ts)
    if ks == 3:
        out_c = C
        table_ref = FO.me_lookup(C, out_c, 3, ts)
    else:  # stride-2 downsampling conv: outputs on the 2*ts lattice
        oc = C.copy(); oc[:, 1:] = oc[:, 1:] // (2 * ts) * (2 * ts)
        out_c = np.unique(oc, axis=0)
        table_ref = FO.me_lookup(C, out_c, 2, ts)
    keys, vals = ops.hash_build(torch.from_numpy(C).cuda())
    table = ops.kmap_lookup(keys, vals, torch.from_numpy(out_c).cuda(), (ks,) * 3, (ts,) * 3, convention=1)
    assert (table.cpu().numpy() == table_ref).all()
    f = torch.from_numpy(rng.normal(0, 1, (C.shape[0], cin)).astype(np.float32)).to(dtype)
    w = torch.from_numpy((rng.normal(0, 1, (ks ** 3, cin, cout)) / np.sqrt(cin * 4)).astype(np.float32)).to(dtype)
    b = rng.normal(0, 0.1, cout).astype(np.float32)
    want = FO.act(FO.sparse_conv_f32(f.float().numpy(), w.float().numpy(), table_ref, b), 'relu')
    got = ops.spconv_f16(f.cuda(), w.permute(0, 2, 1).contiguous().cuda(), table, bias=torch.from_numpy(b).cuda(), act=ops.ACT_RELU)
    assert got.dtype == dtype
    assert _rel(got.float().cpu().numpy(), want) < TOL[dtype]
    # residual + post activation (ResBlock tail), fp32 output
    res = torch.from_numpy(rng.normal(0, 1, (out_c.shape[0], cout)).astype(np.float32))
    want2 = FO.act(FO.sparse_conv_f32(f.float().numpy(), w.float().numpy(), table_ref, b) + res.numpy(), 'leaky_relu', 0.2)
    got2 = ops.spconv_f16(f.cuda(), w.permute(0, 2, 1).contiguous().cuda(), table, bias=torch.from_numpy(b).cuda(),
                          residual=res.cuda(), post_act=ops.ACT_LEAKY, post_slope=0.2, out_dtype=torch.float32)
    assert _rel(got2.cpu().numpy(), want2) < TOL[dtype]
    # determinism: the same launch twice gives identical bits (encoder/decoder of a float codec rely on it)
    again = ops.spconv_f16(f.cuda(), w.permute(0, 2, 1).contiguous().cuda(), table, bias=torch.from_numpy(b).cuda(), act=ops.ACT_RELU)
    assert torch.equal(got, again)
    # rows regrouped by neighbour pattern: skipped offsets only ever contributed exact zeros, so the bits are the same
    tp, perm = ops.group_rows(table)
    grouped = ops.spconv_f16(f.cuda(), w.permute(0, 2, 1).contiguous().cuda(), tp, bias=torch.from_numpy(b).cuda(),
                             residual=res.cuda(), post_act=ops.ACT_LEAKY, post_slope=0.2, out_dtype=torch.float32, row_perm=perm)
    assert torch.equal(grouped, got2)


@pytest.mark.parametrize('dtype', [torch.float16, torch.bfloat16])
def test_linear_f16_and_selected_children(dtype):
    from fastpcc_b200 import ops
    rng = np.random.default_rng(3)
    m, k, n = 3000, 128, 64
    a = torch.from_numpy(rng.normal(0, 1, (m, k)).astype(np.float32)).to(dtype)
    w = torch.from_numpy((rng.normal(0, 1, (n, k)) / np.sqrt(k)).astype(np.float32)).to(dtype)
    b = rng.normal(0, 0.1, n).astype(np.float32)
    want = a.float().numpy() @ w.float().numpy().T + b
    got = ops.linear_f16(a.cuda(), w.cuda(), bias=torch.from_numpy(b).cuda())
    assert _rel(got.float().cpu().numpy(), want) < TOL[dtype]
    # transposed conv k2 s2 onto existing children == one weight block per child slot (selection linear)
    occ = rng.integers(1, 256, m).astype(np.uint8)
    w8 = torch.from_numpy((rng.normal(0, 1, (8 * n, k)) / np.sqrt(k)).astype(np.float32)).to(dtype)
    coords = torch.from_numpy(synth.with_batch(np.stack([np.arange(m), np.zeros(m), np.zeros(m)], 1).astype(np.int32))).cuda()
    _, par, slot, nchild = ops.upsample(coords, torch.from_numpy(occ).cuda(), want_coords=False)
    sel = ops.slot_pairs(par, slot)
    got = ops.linear_f16(a.cuda(), w8.cuda(), sel=sel, n_out_rows=nchild).float().cpu().numpy()
    dense = (a.float().numpy() @ w8.float().numpy().T).reshape(m, 8, n)
    bits = ((occ[:, None] >> np.arange(7, -1, -1)[None]) & 1).astype(bool)
    assert _rel(got, dense[bits]) < TOL[dtype]


def test_torchsparse_style_layers_match_fp32_reference():
    """fastpcc_b200.torchsparse_nn (Conv3d / functional conv3d / Block of lossl_coord/model.py:34-46,356-374,645-660)
    against the fp32 oracle on the reference's own kernel-map convention (hashmap_cuda.cuh:221-275), incl. the strided
    2x2x2 `get_bin` convolution with an explicit weight."""
    from fastpcc_b200 import synth, torchsparse_nn as TS
    from fastpcc_b200.sparse_tensor import SparseTensor
    from oracle import int_ops as K
    rng = np.random.default_rng(21)
    xyz = synth.surface_cloud(4, bits=7, n_target=6000)
    C = synth.with_batch(xyz)
    C = C[np.lexsort((C[:, 3], C[:, 2], C[:, 1], C[:, 0]))]
    ch = 32
    f = rng.normal(0, 1, (C.shape[0], ch)).astype(np.float32)
    x = SparseTensor(torch.from_numpy(f).cuda().half(), torch.from_numpy(C).cuda(), 1)
    blk = TS.Block(ch).cuda()
    with torch.no_grad():
        blk.act.weight.fill_(0.2)
        blk.act2.weight.fill_(0.1)
    with torch.no_grad():                                                      # inference: fused epilogues
        got = blk(x).F.float().cpu().numpy()
    table = K.lookup_coords(C, C, (3, 3, 3), (1, 1, 1))                        # [K, n], input row + 1, 0 = none
    f16 = x.F.float().cpu().numpy()
    w1, w2 = (m.kernel.detach().half().float().cpu().numpy() for m in (blk.conv, blk.conv2))
    b1, b2 = (m.bias.detach().float().cpu().numpy() for m in (blk.conv, blk.conv2))
    h = FO.act(FO.sparse_conv_f32(f16, w1, table, b1), 'leaky_relu', 0.2).astype(np.float16).astype(np.float32)
    want = FO.act(FO.sparse_conv_f32(h, w2, table, b2) + f16, 'leaky_relu', 0.1)
    assert _rel(got, want) < TOL[torch.float16]
    # get_bin: ones features, fold kernel 2x2x2 stride 2 with an explicit [8, 1, 1] weight of powers of two
    ones = SparseTensor(torch.ones((C.shape[0], 1), device='cuda'), torch.from_numpy(C).cuda(), 1)
    fold = torch.tensor([128., 64., 32., 16., 8., 4., 2., 1.], device='cuda').reshape(8, 1, 1)
    ret = TS.conv3d(ones, weight=fold, kernel_size=(2, 2, 2), bias=None, stride=(2, 2, 2), out_dtype=torch.float32)
    Cp = np.unique(np.concatenate([C[:, :1], C[:, 1:] >> 1], 1), axis=0)
    assert (ret.C.cpu().numpy() == Cp).all() and ret.stride == (2, 2, 2)
    tb = K.lookup_coords(C, Cp, (2, 2, 2), (2, 2, 2))
    occ = ((tb != 0) * fold.reshape(8, 1).cpu().numpy()).sum(0)
    assert (ret.F.cpu().numpy()[:, 0] == occ).all()                            # exact: small integers in fp16 / fp32


def test_conv3d_autograd_matches_dense_reference():
    """Training slice (SURVEY §8a row 19): gradients of the fused sparse conv (`torchsparse_nn.conv3d` with an explicit
    weight and bias) w.r.t. features, weights and bias against torch autograd through the same sum written with
    index_select + matmul in fp32, for the conv and the 1x1 (linear) kinds; then a Block trains one SGD step."""
    from fastpcc_b200 import synth, ops, torchsparse_nn as TS
    from fastpcc_b200.sparse_tensor import SparseTensor
    rng = np.random.default_rng(8)
    C = synth.with_batch(synth.surface_cloud(6, bits=7, n_target=3000))
    C = torch.from_numpy(C[np.lexsort((C[:, 3], C[:, 2], C[:, 1], C[:, 0]))]).cuda()
    n, cin, cout = C.shape[0], 24, 40
    keys, vals = ops.hash_build(C)
    for ks, st, out_c in (((3, 3, 3), (1, 1, 1), C), ((1, 1, 1), (1, 1, 1), C),
                          ((2, 2, 2), (2, 2, 2), torch.unique(torch.cat([C[:, :1], C[:, 1:] >> 1], 1), dim=0))):
        table = ops.kmap_lookup(keys, vals, out_c.contiguous(), ks, st)
        kv = table.shape[0]
        a = torch.randn(n, cin, device='cuda').half().float().requires_grad_()
        w = (torch.randn(kv, cin, cout, device='cuda') / (kv * cin) ** 0.5).half().float().requires_grad_()
        b = torch.randn(cout, device='cuda').requires_grad_()
        gout = torch.randn(table.shape[1], cout, device='cuda').half().float()
        ret = TS.conv3d(SparseTensor(a, C, 1), w, ks, bias=b, stride=st)
        assert torch.equal(ret.C, out_c)                                    # the rows of `table`
        out = ret.F
        out.backward(gout)
        got = (out.detach(), a.grad.clone(), w.grad.clone(), b.grad.clone())
        a.grad = w.grad = b.grad = None
        a_pad = torch.cat([torch.zeros(1, cin, device='cuda'), a])          # row 0 = "no neighbour"
        ref = sum(a_pad[table[k].long()] @ w[k] for k in range(kv)) + b
        ref.backward(gout)
        for g_, r_, name in zip(got, (ref.detach(), a.grad, w.grad, b.grad), ('out', 'd_feats', 'd_weight', 'd_bias')):
            err = float((g_ - r_).abs().max() / r_.abs().max().clamp(min=1e-6))
            assert err < 1e-2, (ks, name, err)
    blk = TS.Block(32).cuda()
    x = SparseTensor(torch.randn(n, 32, device='cuda'), C, 1)
    opt = torch.optim.SGD(blk.parameters(), lr=1e-2)
    losses = []
    for _ in range(3):
        opt.zero_grad()
        loss = blk(x).F.float().pow(2).mean()
        loss.backward()
        opt.step()
        losses.append(float(loss.detach()))
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in blk.parameters())
    assert losses[-1] < losses[0]


@pytest.mark.parametrize('cin,cout,dt', [(128, 128, torch.float16), (256, 192, torch.bfloat16), (64, 256, torch.float16), (24, 40, torch.float16)])
def test_tensor_core_wgrad_equals_per_offset_gemm(cin, cout, dt):
    """fpcc_spconv_wgrad_f16 (tcgen05, both operands MN-major, split-K tiles meeting in fp32 atomics) against the
    per-offset gather + fp32 matmul it replaces, on the 3x3x3 map of a surface cloud (tiles of one offset larger and
    smaller than 2048 pairs, offsets without pairs on the strided map).  Tolerance: fp32 accumulation of exact
    fp16 / bf16 products in a different order, 1e-3 of the largest entry."""
    from fastpcc_b200 import synth, ops
    C = synth.with_batch(synth.surface_cloud(6, bits=8, n_target=12000))
    C = torch.from_numpy(C[np.lexsort((C[:, 3], C[:, 2], C[:, 1], C[:, 0]))]).cuda()
    keys, vals = ops.hash_build(C)
    for ks, st, out_c in (((3, 3, 3), (1, 1, 1), C),
                          ((2, 2, 2), (2, 2, 2), torch.unique(torch.cat([C[:, :1], C[:, 1:] >> 1], 1), dim=0))):
        table = ops.kmap_lookup(keys, vals, out_c.contiguous(), ks, st)
        kv = table.shape[0]
        x = torch.randn(C.shape[0], cin, device='cuda').to(dt)
        g = torch.randn(table.shape[1], cout, device='cuda').to(dt)
        in_map, out_map, offsets = ops.kmap_compact(table)
        off = offsets.tolist()
        got = ops.spconv_wgrad_f16(x, g, in_map, out_map, off, cin, cout)
        want = torch.zeros((kv, cin, cout), dtype=torch.float32, device='cuda')
        for k in range(kv):
            s_, e_ = off[k], off[k + 1]
            if e_ > s_:
                want[k] = x.float()[in_map[s_:e_].long()].t() @ g.float()[out_map[s_:e_].long()]
        err = float((got - want).abs().max() / want.abs().max())
        assert got.shape == want.shape and err < 1e-3, (ks, cin, cout, err)

