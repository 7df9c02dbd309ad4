"""Training support for the float sparse convolution (SURVEY §8a row 19): torch.autograd.Functions around the tcgen05
kernels, shared by the torchsparse-shaped layers (`torchsparse_nn.py`) and the MinkowskiEngine shim (`me.py`).

  forward   out[m]  = act(sum_k  A[nbr_k(m)] @ W[k] + bias)          fused tcgen05 kernel, fp32 accumulation
  act'      dZ      = dOut * act'(out), dbias = sum_m dZ[m]          `fpcc_act_grad_f16`: one pass, read from the
                                                                    forward output (ReLU / LeakyReLU with slope >= 0)
  dgrad     dA[j]   = sum_k  dZ[nbr_k^T(j)] @ W[k]^T                 the SAME kernel on the transposed kernel map
                                                                    (`fpcc_kmap_transpose`, no host sync): the
                                                                    parameter layout [K, C_in, C_out] is exactly the
                                                                    [K, C_out', C_in'] operand the kernel wants
  wgrad     dW[k]   = A[in_k]^T @ dZ[out_k]                          `fpcc_spconv_wgrad_f16`: tcgen05 with BOTH operands
                                                                    MN-major (the contraction runs over the gathered
                                                                    rows), split-K tiles meeting in fp32 atomics; a
                                                                    per-offset library GEMM only above 256 channels

The deep-factorized entropy model (`FactorizedBitsFunction`) is one fused kernel each way: bits of the latents forward,
dy and the packed parameter gradient backward (`fpcc_factorized_bits` / `fpcc_factorized_grad`).

MinkowskiEngine computes the same three products per kernel offset (ME backward = transposed gather-GEMM-scatter).
The ME layer kinds map onto these products as follows (`MELayerFunction`):

  conv   kv > 1 (stride 1, k2s2, explicit target key)   dgrad on kmap_transpose(table), wgrad on kmap_compact(table)
  linear 1x1 conv, MinkowskiLinear                      dgrad linear_f16(dZ, W^T), wgrad with kv = 1 identity pairs
  tconv  k2s2 onto an existing key (selection linear)   the conv rules on the child-slot table [8, n_child]
  gen    generative k2s2 (dense C_in -> 8 C_out)        dgrad linear_f16(dZ.view(N, 8 C_out'), W8^T), wgrad with
                                                        kv = 8 and pairs (n -> 8n + k)
"""
import torch

from . import ops

WGRAD_TC = True  # False: per-offset library GEMMs (A/B switch for the tests)


def transpose_table(table: torch.Tensor, n_in: int) -> torch.Tensor:
    """k-major map of the transposed convolution: tt[k, j] = m + 1 where table[k, m] == j + 1 (0 = none).  Each
    (offset, input row) pairs with at most one output row, so the scatter has no collisions (fpcc_kmap_transpose)."""
    return ops.kmap_transpose(table, n_in)


# Tensors derived from a kernel map (transposed map for dgrad, compacted pair lists + tile offsets for wgrad) are the same
# for every layer and every step that uses the map: built once per table.  The entry keeps the table itself alive, so its
# address cannot be reused by another tensor while the entry exists; a handful of maps are live at a time.
_derived_cache = {}
_DERIVED_MAX = 64


def _derived(table: torch.Tensor, n_in: int) -> dict:
    key = (table.data_ptr(), tuple(table.shape), n_in, table.device.index)
    ent = _derived_cache.get(key)
    if ent is None:
        if len(_derived_cache) >= _DERIVED_MAX:
            _derived_cache.pop(next(iter(_derived_cache)))
        ent = {'table': table}
        _derived_cache[key] = ent
    return ent


def _transposed(table, n_in):
    ent = _derived(table, n_in)
    if 'tt' not in ent:
        ent['tt'] = transpose_table(table, n_in)
    return ent['tt']


def _transposed_grouped(table, n_in):
    """(transposed table regrouped by neighbour pattern, row permutation): the dgrad's twin of the forward's grouping"""
    ent = _derived(table, n_in)
    if 'tt_grouped' not in ent:
        ent['tt_grouped'] = ops.group_rows(_transposed(table, n_in))
    return ent['tt_grouped']


def _compacted(table, n_in):
    ent = _derived(table, n_in)
    if 'pairs' not in ent:
        in_map, out_map, offsets = ops.kmap_compact(table)
        ent['pairs'] = (in_map, out_map, offsets.tolist())
    return ent['pairs']


def _wgrad(x, dz, in_map, out_map, off, c_in, c_out):
    """dW[k] = x[in_k]^T @ dz[out_k] -> fp32 [kvol, c_in, c_out]; x [n_in, >= c_in], dz [n_out, >= c_out] compute dtype"""
    if WGRAD_TC and ops.wgrad_supported(c_in, c_out):
        # tensor cores: contraction over the gathered rows, both operands MN-major (fpcc_spconv_wgrad_f16)
        return ops.spconv_wgrad_f16(x, dz, in_map, out_map, off, c_in, c_out)
    # library GEMM per offset (wide layers)
    a32, g32 = x[:, :c_in].float(), dz[:, :c_out].float()
    dw = torch.zeros((len(off) - 1, c_in, c_out), dtype=torch.float32, device=x.device)
    for k in range(len(off) - 1):
        s, e = off[k], off[k + 1]
        if e > s:
            dw[k] = a32[in_map[s:e].long()].t() @ g32[out_map[s:e].long()]
    return dw


class SparseConvFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feats, weight, bias, table, compute_dtype):
        kv, c_in, c_out = weight.shape
        cin_p, cout_p = max(16, (c_in + 7) // 8 * 8), max(16, c_out)
        f = torch.nn.functional.pad(feats.to(compute_dtype), (0, cin_p - c_in)).contiguous()
        w_t = torch.zeros((kv, cout_p, cin_p), dtype=compute_dtype, device=weight.device)
        w_t[:, :c_out, :c_in] = weight.detach().permute(0, 2, 1).to(compute_dtype)
        b = None
        if bias is not None:
            b = torch.zeros(cout_p, dtype=torch.float32, device=weight.device)
            b[:c_out] = bias.detach().float().reshape(-1)
        out = ops.spconv_f16(f, w_t, table, bias=b, out_dtype=torch.float32)[:, :c_out]
        ctx.save_for_backward(feats, weight, table)
        ctx.has_bias, ctx.compute_dtype = bias is not None, compute_dtype
        return out.to(feats.dtype if feats.dtype.is_floating_point else torch.float32)

    @staticmethod
    def backward(ctx, grad_out):
        feats, weight, table = ctx.saved_tensors
        kv, c_in, c_out = weight.shape
        dt = ctx.compute_dtype
        g = grad_out.contiguous()
        d_feats = d_weight = d_bias = None
        if ctx.needs_input_grad[0]:
            cin_p, cout_p = max(16, c_in), max(16, (c_out + 7) // 8 * 8)
            gp = torch.nn.functional.pad(g.to(dt), (0, cout_p - c_out)).contiguous()
            w = torch.zeros((kv, cin_p, cout_p), dtype=dt, device=weight.device)   # [K, "C_out" = c_in, "C_in" = c_out]
            w[:, :c_in, :c_out] = weight.detach().to(dt)
            tt = _transposed(table, feats.shape[0])
            d_feats = ops.spconv_f16(gp, w, tt, out_dtype=torch.float32)[:, :c_in].to(feats.dtype)
        if ctx.needs_input_grad[1]:
            in_map, out_map, off = _compacted(table, feats.shape[0])
            d_weight = _wgrad(feats.to(dt), g.to(dt), in_map, out_map, off, c_in, c_out).to(weight.dtype)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            d_bias = g.float().sum(0)
        return d_feats, d_weight, d_bias, None, None


def sparse_conv(feats, weight, bias, table, compute_dtype=torch.float16):
    """differentiable sparse convolution: feats [n_in, C_in], weight [K, C_in, C_out], k-major table [K, n_out]"""
    return SparseConvFunction.apply(feats, weight, bias, table, compute_dtype)


class MESpec:
    """What the backward of one MinkowskiEngine-shim layer needs (built by `me.py`, which owns the forward):
    kind 'conv' | 'linear' | 'tconv' | 'gen'; table: the UNGROUPED k-major map (conv) or the child-slot table (tconv);
    group: regroup the transposed table (the forward's GROUP_ROWS_MIN rule on the dgrad's output rows); layout of the
    kernel parameter: 'kio' [K, C_in, C_out], 'io' [C_in, C_out] (1x1 conv), 'oi' [C_out, C_in] (nn.Linear); dtype: the
    compute dtype of the forward, in which the feature gradients travel."""

    def __init__(self, kind, c_in, c_out, act, slope, dtype, layout='kio', table=None, group=False):
        self.kind, self.c_in, self.c_out, self.act, self.slope, self.dtype = kind, c_in, c_out, act, slope, dtype
        self.layout, self.table, self.group = layout, table, group


def _kio(kernel, layout):
    w = kernel.detach().float()
    return w if layout == 'kio' else (w[None] if layout == 'io' else w.t()[None])


class MELayerFunction(torch.autograd.Function):
    """One conv / linear layer of the ME shim with its fused epilogue (bias, ReLU / LeakyReLU slope >= 0).  The forward
    is the layer's own inference call (`run`), so the output bits do not depend on the grad mode."""

    @staticmethod
    def forward(ctx, feats, kernel, bias, spec, run):
        y = run()
        ctx.spec = spec
        ctx.bias_shape = None if bias is None else bias.shape
        ctx.save_for_backward(feats, kernel, y)
        return y

    @staticmethod
    def backward(ctx, dy):
        feats, kernel, y = ctx.saved_tensors
        sp = ctx.spec
        need_x, need_w = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        need_b = ctx.bias_shape is not None and ctx.needs_input_grad[2]
        dt = sp.dtype
        c_in, c_out = sp.c_in, sp.c_out
        c_pad = max(16, (c_out + 7) // 8 * 8)  # operand width of the dgrad / wgrad kernels
        dz, db = ops.act_grad_f16(dy, y, sp.act, sp.slope, c_pad, out_dtype=dt, want_bias=need_b)
        w = _kio(kernel, sp.layout)  # fp32 [K, C_in, C_out]
        kv = w.shape[0]
        d_feats = d_kernel = d_bias = None
        n_in = feats.shape[0]
        if need_x:
            cin_o = max(16, c_in)
            if sp.kind in ('conv', 'tconv'):
                wd = torch.zeros((kv, cin_o, c_pad), dtype=dt, device=w.device)  # [K, "C_out" = c_in, "C_in" = c_out]
                wd[:, :c_in, :c_out] = w.to(dt)
                if sp.group:
                    tt, perm = _transposed_grouped(sp.table, n_in)
                else:
                    tt, perm = _transposed(sp.table, n_in), None
                d_feats = ops.spconv_f16(dz, wd, tt, out_dtype=dt, row_perm=perm)
            elif sp.kind == 'linear':
                wl = torch.zeros((cin_o, c_pad), dtype=dt, device=w.device)
                wl[:c_in, :c_out] = w[0].to(dt)
                d_feats = ops.linear_f16(dz, wl, out_dtype=dt)
            else:  # gen: the 8 children of row n are rows 8n..8n+7 of dZ, i.e. one row of dZ.view(N, 8 c_pad)
                wg = torch.zeros((cin_o, 8, c_pad), dtype=dt, device=w.device)
                wg[:c_in, :, :c_out] = w.permute(1, 0, 2).to(dt)
                d_feats = ops.linear_f16(dz.view(n_in, 8 * c_pad), wg.reshape(cin_o, 8 * c_pad), out_dtype=dt)
            d_feats = d_feats[:, :c_in] if d_feats.shape[1] != c_in else d_feats
        if need_w:
            x = feats.to(dt).contiguous()
            if sp.kind in ('conv', 'tconv'):
                in_map, out_map, off = _compacted(sp.table, n_in)
            elif sp.kind == 'linear':
                in_map = torch.arange(n_in, dtype=torch.int32, device=x.device)
                out_map, off = in_map, [0, n_in]
            else:
                r = torch.arange(n_in, dtype=torch.int32, device=x.device)
                in_map = r.repeat(8)
                out_map = (8 * r[None] + torch.arange(8, dtype=torch.int32, device=x.device)[:, None]).reshape(-1)
                off = [k * n_in for k in range(9)]
            dw = _wgrad(x, dz, in_map, out_map, off, c_in, c_out)
            d_kernel = dw if sp.layout == 'kio' else (dw[0] if sp.layout == 'io' else dw[0].t())
        if need_b:
            d_bias = db.reshape(ctx.bias_shape)
        return d_feats, d_kernel, d_bias, None, None


def me_layer(feats, kernel, bias, spec, run):
    """differentiable ME-shim layer: `run()` computes the forward output from `feats` with the layer's inference kernels"""
    return MELayerFunction.apply(feats, kernel, bias, spec, run)


class FactorizedBitsFunction(torch.autograd.Function):
    """bits = -log2(max(L(y), bound)) of the deep-factorized prior (fpcc_factorized_bits): y fp32 [n, C], params fp32
    [C, 43] (the packed rows of `entropy_models.NoisyDeepFactorizedEntropyModel`).  The backward recomputes the
    forward in the kernel and returns the gradient of the raw params, reduced in a fixed order."""

    @staticmethod
    def forward(ctx, y, params, bound):
        ctx.save_for_backward(y, params)
        ctx.bound = bound
        return ops.factorized_bits(y, params, bound)

    @staticmethod
    def backward(ctx, dbits):
        y, params = ctx.saved_tensors
        dy, dp = ops.factorized_grad(y, params, dbits.float(), ctx.bound)
        return (dy if ctx.needs_input_grad[0] else None), (dp if ctx.needs_input_grad[1] else None), None


def factorized_bits(y, params, bound=1e-9):
    """differentiable bits of the deep-factorized prior; y is cast to fp32 (latents arrive in the compute dtype)"""
    return FactorizedBitsFunction.apply(y.float(), params, float(bound))
