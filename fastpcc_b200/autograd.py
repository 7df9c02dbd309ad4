"""Training support for the float sparse convolution (SURVEY §8a row 19): torch.autograd.Functions around the tcgen05
kernels.  Every float conv / linear layer, of the torchsparse-shaped layers (`torchsparse_nn.py`) and of the
MinkowskiEngine shim (`me.py`) alike, trains through `MELayerFunction`: its forward is the layer's own inference call.

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
The Gaussian conditional model of the hyperprior (`GaussianBitsFunction`) likewise: bits forward, dy, dmu and dsigma
backward (`fpcc_gaussian_bits` / `fpcc_gaussian_grad`).

MinkowskiEngine computes the same three products per kernel offset (ME backward = transposed gather-GEMM-scatter).
The layer kinds map onto these products as follows (`MELayerFunction`):

  conv   kv > 1 (stride 1, k2s2, explicit target key)   dgrad on kmap_transpose(table), wgrad on kmap_compact(table)
         (torchsparse: every conv but 1x1 at stride 1)
  linear 1x1 conv, MinkowskiLinear                      dgrad linear_f16(dZ, W^T), wgrad with kv = 1 identity pairs
  tconv  k2s2 onto an existing key (selection linear)   the conv rules on the child-slot table [8, n_child]
  gen    generative k2s2 (dense C_in -> 8 C_out)        dgrad linear_f16(dZ.view(N, 8 C_out'), W8^T), wgrad with
                                                        kv = 8 and pairs (n -> 8n + k)
"""
import torch

from . import ops

WGRAD_TC = True  # False: per-offset library GEMMs (A/B switch for the tests)


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
        ent['tt'] = ops.kmap_transpose(table, n_in)
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


class MESpec:
    """What the backward of one layer needs (built by `me.py` or `torchsparse_nn.py`, which own the forward):
    kind 'conv' | 'linear' | 'tconv' | 'gen'; table: the UNGROUPED k-major map (conv) or the child-slot table (tconv);
    group: regroup the transposed table (the forward's GROUP_ROWS_MIN rule on the dgrad's output rows); layout of the
    kernel parameter: 'kio' [K, C_in, C_out], 'io' [C_in, C_out] (1x1 conv), 'oi' [C_out, C_in] (nn.Linear); dtype: the
    compute dtype of the forward, in which the feature gradients travel (fp32 for fp32 input features)."""

    def __init__(self, kind, c_in, c_out, act, slope, dtype, layout='kio', table=None, group=False):
        self.kind, self.c_in, self.c_out, self.act, self.slope, self.dtype = kind, c_in, c_out, act, slope, dtype
        self.layout, self.table, self.group = layout, table, group


def _kio(kernel, layout):
    w = kernel.detach().float()
    return w if layout == 'kio' else (w[None] if layout == 'io' else w.t()[None])


class MELayerFunction(torch.autograd.Function):
    """One float conv / linear layer with its fused epilogue (bias, ReLU / LeakyReLU slope >= 0).  The forward
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
        c_pad = ops.f16_widths(c_out, c_in)[0]  # dgrad / wgrad reduce over the layer's outputs: the forward's roles swapped
        dz, db = ops.act_grad_f16(dy, y, sp.act, sp.slope, c_pad, out_dtype=dt, want_bias=need_b)
        w = _kio(kernel, sp.layout)  # fp32 [K, C_in, C_out]
        d_feats = d_kernel = d_bias = None
        n_in = feats.shape[0]
        if need_x:
            wd = ops.f16_weight(w.transpose(1, 2), dt)  # [K, "C_out" = c_in, "C_in" = c_out], padded
            dx_dt = torch.float32 if feats.dtype == torch.float32 else dt  # fp32 features get fp32 gradients
            if sp.kind in ('conv', 'tconv'):
                if sp.group:
                    tt, perm = _transposed_grouped(sp.table, n_in)
                else:
                    tt, perm = _transposed(sp.table, n_in), None
                d_feats = ops.spconv_f16(dz, wd, tt, out_dtype=dx_dt, row_perm=perm)
            elif sp.kind == 'linear':
                d_feats = ops.linear_f16(dz, wd[0], out_dtype=dx_dt)
            else:  # gen: the 8 children of row n are rows 8n..8n+7 of dZ, i.e. one row of dZ.view(N, 8 c_pad)
                wg = wd.permute(1, 0, 2).reshape(wd.shape[1], 8 * c_pad)
                d_feats = ops.linear_f16(dz.view(n_in, 8 * c_pad), wg, out_dtype=dx_dt)
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
    """differentiable float layer: `run()` computes the forward output from `feats` with the layer's inference kernels"""
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


class GaussianBitsFunction(torch.autograd.Function):
    """bits = -log2(max(L, bound)) of the Gaussian conditional model (fpcc_gaussian_bits): y, scales, means fp32 [n, C]
    (means None: mean 0; means and scales may be column slices of one tensor).  The backward recomputes the forward in
    the kernel and returns dy, dscales and dmeans."""

    @staticmethod
    def forward(ctx, y, scales, means, scale_bound, bound):
        ctx.save_for_backward(y, scales, means)
        ctx.scale_bound, ctx.bound = scale_bound, bound
        return ops.gaussian_bits(y, scales, means, scale_bound, bound)

    @staticmethod
    def backward(ctx, dbits):
        y, scales, means = ctx.saved_tensors
        need = ctx.needs_input_grad
        dy, dm, ds = ops.gaussian_grad(y, scales, dbits.float(), means, ctx.scale_bound, ctx.bound, need_dmu=need[2])
        return (dy if need[0] else None), (ds if need[1] else None), (dm if need[2] else None), None, None


def gaussian_bits(y, scales, means=None, scale_bound=0.11, likelihood_bound=1e-9):
    """differentiable bits of the Gaussian conditional model; y, scales and means are cast to fp32 (they arrive in the
    shim's compute dtype)"""
    return GaussianBitsFunction.apply(y.float(), scales.float(), None if means is None else means.float(),
                                      float(scale_bound), float(likelihood_bound))
