"""Float (fp16 / bf16 on tcgen05, fp32 accumulation) twin of the torchsparse layer surface that the reference's
floating-point LiDAR codec is written against (models/convolutional/lossl_coord/model.py:34-46,137-175,356-374,
645-672): `Conv3d` (= torchsparse.nn.Conv3d), `conv3d` (= torchsparse.nn.functional.conv3d with an explicit weight,
as used by `get_bin`), `Block`, `SparseSequential`.

Conventions follow torchsparse 2.1 with kmap_mode = 'hashmap' (lossl_coord/model.py:309-312): parameter `kernel` is
[K, C_in, C_out] ([C_in, C_out] when K == 1), the kernel-offset order is the one of the reference's own copy of the
torchsparse hash map (lib/int_sparse_conv/src/hashmap/hashmap_cuda.cuh:221-275: odd kernels x fastest and centred,
even kernels z fastest), a strided conv with kernel == stride writes to coordinates >> log2(stride), and kernel
maps / hash tables are cached on the tensor's `_caches` exactly like the integer layers do, so both families share
them.  Every conv is ONE fused kernel (`fpcc_spconv_f16`, rows grouped by neighbour pattern for large inputs);
activations / residual adds that follow can ride in its epilogue (`fused_act`, `residual`).  Training runs the same
call inside `autograd.MELayerFunction`, the backward the MinkowskiEngine shim's layers train on; there activations and
residual adds stay torch ops."""
import math
from typing import Optional, Tuple, Union

import torch
import torch.nn as nn

from . import autograd, ops
from .int_sparse_conv.cuda_ops import GROUP_ROWS_MIN, KernelMap, build_kernel_map
from .sparse_tensor import SparseTensor, _triple

_COMPUTE = torch.float16


def set_compute_dtype(dtype):
    global _COMPUTE
    assert dtype in (torch.float16, torch.bfloat16)
    _COMPUTE = dtype


def _out_coords(x: SparseTensor, stride: Tuple[int, int, int]):
    if stride == (1, 1, 1):
        return x.stride, x.C
    out_stride = tuple(a * b for a, b in zip(x.stride, stride))
    if out_stride in x._caches.cmaps:
        return out_stride, x._caches.cmaps[out_stride][0]
    assert stride[0] == stride[1] == stride[2] and stride[0] & (stride[0] - 1) == 0, 'power-of-two isotropic strides only'
    c = x.C.clone()
    c[:, 1:] >>= stride[0].bit_length() - 1
    return out_stride, torch.unique(c, dim=0)


def _kernel_map(input: SparseTensor, out_c: torch.Tensor, ks, st) -> KernelMap:
    caches = input._caches
    tag = (input.stride, ks, st)
    entry = caches.kmaps.get(tag)
    kmap = entry.get('in_out_maps') if entry is not None else None
    if not isinstance(kmap, KernelMap):
        kmap, hk = build_kernel_map(input.C, out_c, ks, st, caches.hashmaps.get(input.stride))
        caches.hashmaps.setdefault(input.stride, hk)
        caches.kmaps.setdefault(tag, {})['in_out_maps'] = kmap
    return kmap


def conv3d(input: SparseTensor, weight: torch.Tensor, kernel_size=3, bias: Optional[torch.Tensor] = None, stride=1,
           padding=0, dilation=1, transposed: bool = False, generative: bool = False, config=None, training: bool = False,
           fused_act: int = ops.ACT_NONE, slope: float = 0.0, residual: Optional[torch.Tensor] = None,
           post_act: int = ops.ACT_NONE, post_slope: float = 0.0, out_dtype=None, _weight_t=None) -> SparseTensor:
    """torchsparse.nn.functional.conv3d (non-transposed): weight [K, C_in, C_out] or [C_in, C_out].
    With grad enabled and the weight or the features requiring it, the same call runs inside `autograd.me_layer`, which
    gives it its backward: the output then leaves in the features' float dtype (fp32 for other features), and fused
    activations and residuals are refused (they follow as torch ops)."""
    assert not transposed and not generative, 'the codec path uses forward convolutions only'
    assert _triple(dilation) == (1, 1, 1)
    ks, st = _triple(kernel_size), _triple(stride)
    kv = math.prod(ks)
    w = weight[None] if weight.dim() == 2 else weight
    assert w.shape[0] == kv, f'weight has {w.shape[0]} offsets, kernel {ks} needs {kv}'
    c_in, c_out = w.shape[1], w.shape[2]
    cin_p, cout_p = ops.f16_widths(c_in, c_out)
    training = torch.is_grad_enabled() and (weight.requires_grad or input.F.requires_grad)
    if training:
        assert fused_act == ops.ACT_NONE and residual is None and post_act == ops.ACT_NONE, 'fused epilogues are inference only'
        out_dtype = input.F.dtype if input.F.dtype.is_floating_point else torch.float32
    if _weight_t is None:
        _weight_t = ops.f16_weight(w, _COMPUTE)
    b = None
    if bias is not None:
        b = torch.zeros(cout_p, dtype=torch.float32, device=w.device)
        b[:c_out] = bias.detach().reshape(-1).float()
    f = ops.pad_cols(input.F.to(_COMPUTE), cin_p).contiguous()
    if residual is not None:
        residual = ops.pad_cols(residual.to(out_dtype or _COMPUTE), cout_p).contiguous()
    out_stride, out_c = _out_coords(input, st)
    linear = kv == 1 and st == (1, 1, 1)
    kmap = None if linear else _kernel_map(input, out_c, ks, st)

    def run():
        if linear:
            out = ops.linear_f16(f, _weight_t[0], bias=b, act=fused_act, slope=slope, residual=residual, post_act=post_act,
                                 post_slope=post_slope, out_dtype=out_dtype)
        else:
            if kmap.table.shape[1] >= GROUP_ROWS_MIN:
                table, perm = kmap.grouped()
            else:
                table, perm = kmap.table, None
            out = ops.spconv_f16(f, _weight_t, table, bias=b, act=fused_act, slope=slope, residual=residual,
                                 post_act=post_act, post_slope=post_slope, out_dtype=out_dtype, row_perm=perm)
        return out[:, :c_out] if cout_p != c_out else out

    if training:
        sp = autograd.MESpec('linear' if linear else 'conv', c_in, c_out, ops.ACT_NONE, 0.0, _COMPUTE,
                             layout='kio' if weight.dim() == 3 else 'io', table=None if linear else kmap.table,
                             group=input.F.shape[0] >= GROUP_ROWS_MIN)
        out = autograd.me_layer(input.F, weight, bias, sp, run)
    else:
        out = run()
    caches = input._caches
    caches.cmaps.setdefault(input.stride, (input.C, input.spatial_range))
    caches.cmaps.setdefault(out_stride, (out_c, None))
    ret = SparseTensor(out, out_c, out_stride, None)
    ret._caches = caches
    return ret


class Conv3d(nn.Module):
    """torchsparse.nn.Conv3d(in_channels, out_channels, kernel_size, stride, dilation, bias); parameters `kernel`, `bias`."""

    def __init__(self, in_channels: int, out_channels: int, kernel_size: Union[int, Tuple[int, ...]] = 3,
                 stride: Union[int, Tuple[int, ...]] = 1, dilation: int = 1, bias: bool = False, transposed: bool = False,
                 generative: bool = False, **_):
        super().__init__()
        assert not transposed and not generative
        self.in_channels, self.out_channels = in_channels, out_channels
        self.kernel_size, self.stride, self.dilation = _triple(kernel_size), _triple(stride), dilation
        kv = math.prod(self.kernel_size)
        shape = (kv, in_channels, out_channels) if kv > 1 else (in_channels, out_channels)
        self.kernel = nn.Parameter(torch.zeros(shape))
        self.bias = nn.Parameter(torch.zeros(out_channels)) if bias else None
        std = 1.0 / math.sqrt((out_channels if transposed else in_channels) * kv)
        with torch.no_grad():
            self.kernel.uniform_(-std, std)
            if self.bias is not None:
                self.bias.uniform_(-std, std)
        self._cache = None

    def _weight_t(self):
        key = (self.kernel._version, self.kernel.data_ptr(), _COMPUTE)
        if self._cache is None or self._cache[0] != key:
            k = self.kernel.detach()
            w = ops.f16_weight(k[None] if k.dim() == 2 else k, _COMPUTE)
            torch.cuda.current_stream().synchronize()  # the cache may be read from another stream next
            self._cache = (key, w)
        return self._cache[1]

    def forward(self, input: SparseTensor, fused_act: int = ops.ACT_NONE, slope: float = 0.0, residual=None,
                post_act: int = ops.ACT_NONE, post_slope: float = 0.0, out_dtype=None) -> SparseTensor:
        training = torch.is_grad_enabled() and (self.kernel.requires_grad or input.F.requires_grad)
        return conv3d(input, self.kernel, self.kernel_size, self.bias, self.stride, dilation=self.dilation,
                      fused_act=fused_act, slope=slope, residual=residual, post_act=post_act, post_slope=post_slope,
                      out_dtype=out_dtype, _weight_t=None if training else self._weight_t())


class Block(nn.Module):
    """lossl_coord/model.py:645-660: conv - PReLU - conv - (+ input) - PReLU; both activations and the residual add ride
    in the conv epilogues (two kernels instead of two convs + three element-wise passes)."""

    def __init__(self, ch: int):
        super().__init__()
        self.ch = ch
        self.conv = Conv3d(ch, ch, 3, 1, 1, bias=True)
        self.act = nn.PReLU()
        self.conv2 = Conv3d(ch, ch, 3, 1, 1, bias=True)
        self.act2 = nn.PReLU()

    def forward(self, org: SparseTensor) -> SparseTensor:
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            x = self.conv(org)                     # training: the reference's own sequence, autograd through every step
            x.F = self.act(x.F)
            x = self.conv2(x)
            x.F = self.act2(x.F + org.F)
            return x
        x = self.conv(org, fused_act=ops.ACT_LEAKY, slope=float(self.act.weight.detach().reshape(-1)[0]))
        return self.conv2(x, residual=org.F, post_act=ops.ACT_LEAKY, post_slope=float(self.act2.weight.detach().reshape(-1)[0]),
                          out_dtype=org.F.dtype if org.F.dtype in (torch.float16, torch.bfloat16, torch.float32) else None)


class SparseSequential(nn.Sequential):
    """lossl_coord/model.py:663-672"""

    def forward(self, input: SparseTensor) -> SparseTensor:
        x = SparseTensor(input.F, input.C, input.stride, input.spatial_range)
        x._caches = input._caches
        for module in self:
            if isinstance(module, (nn.Linear, nn.LayerNorm, nn.ReLU, nn.LeakyReLU, nn.PReLU)):
                x.F = module(x.F.to(module.weight.dtype) if hasattr(module, 'weight') and module.weight is not None else x.F)
            else:
                x = module(x)
        return x
