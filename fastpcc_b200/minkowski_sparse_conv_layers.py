"""Float layer API, drop-in for lib/minkowski_sparse_conv_layers.py of the reference: same block classes,
constructor signatures, attribute names (`.conv.kernel`, `.conv.kernel_generator.*`, `.mlp.linear.weight`) and
`forward(x, *args)` conventions, on the B200 kernels through the ME-shaped shim `fastpcc_b200.me`.
A block's activation rides in the conv / linear epilogue whenever it is ReLU, LeakyReLU or a single-slope PReLU.
"""
import math
from typing import Any, Callable, Dict, List, Optional, Tuple, Union

import torch
from torch import nn as nn

from . import me as ME


def get_act_module(act: Union[str, nn.Module, None]) -> Optional[nn.Module]:
    """lib/minkowski_sparse_conv_layers.py:10-28"""
    if isinstance(act, nn.Module):
        return act
    if act is None or act == 'None':
        return None
    if act == 'relu':
        return ME.MinkowskiReLU(inplace=True)
    if act.startswith('leaky_relu'):
        return ME.MinkowskiLeakyReLU(negative_slope=float(act.split('(', 1)[1].split(')', 1)[0]), inplace=True)
    if act == 'sigmoid':
        return ME.MinkowskiSigmoid()
    if act == 'prelu':
        return ME.MinkowskiPReLU()
    raise NotImplementedError(act)


def _fusable(act_module) -> bool:
    return ME._fusable_act(act_module)


class MEMLPBlock(nn.Module):
    """:31-53"""

    def __init__(self, in_channels: int, out_channels: int, bn: bool = False, act: Union[str, nn.Module, None] = 'relu'):
        super().__init__()
        self.mlp = ME.MinkowskiLinear(in_channels, out_channels, bias=not bn)
        self.bn = ME.MinkowskiBatchNorm(out_channels) if bn else None
        self.act = get_act_module(act)

    def forward(self, x):
        if self.bn is None and _fusable(self.act):
            return self.mlp(x, fused_act=self.act)
        x = self.mlp(x)
        if self.bn is not None:
            x = self.bn(x)
        if self.act is not None:
            x = self.act(x)
        return x

    def __repr__(self):
        return f'MEMLPBlock(in_ch={self.mlp.linear.in_features}, out_ch={self.mlp.linear.out_features}, ' \
               f'bn={self.bn is not None}, act={self.act})'


class BaseConvBlock(nn.Module):
    """:56-111"""

    def __init__(self, conv_class: Callable, in_channels, out_channels, kernel_size, stride, dilation=1, dimension=3,
                 region_type: str = 'HYPER_CUBE', bn: bool = False, bias: Optional[bool] = None,
                 act: Union[str, nn.Module, None] = 'relu'):
        super().__init__()
        self.region_type = getattr(ME.RegionType, region_type)
        self.conv = conv_class(
            in_channels, out_channels, kernel_size=kernel_size, stride=stride, dilation=dilation,
            bias=bias if bias is not None else not bn,
            kernel_generator=ME.KernelGenerator(kernel_size, stride, dilation, region_type=self.region_type, dimension=dimension),
            dimension=dimension)
        self.bn = ME.MinkowskiBatchNorm(out_channels) if bn else None
        self.act = act
        self.act_module = get_act_module(act)

    def forward(self, x, *args, **kwargs):
        if self.bn is None and _fusable(self.act_module):
            return self.conv(x, *args, fused_act=self.act_module, **kwargs)
        x = self.conv(x, *args, **kwargs)
        if self.bn is not None:
            x = self.bn(x)
        if self.act_module is not None:
            x = self.act_module(x)
        return x

    def __repr__(self):
        kg = self.conv.kernel_generator
        one = lambda t: t[0] if len(set(t)) == 1 else t  # noqa: E731
        return f'{self.conv.__class__.__name__.replace("Minkowski", "ME", 1).replace("Convolution", "Conv", 1)}(' \
               f'in={self.conv.in_channels}, out={self.conv.out_channels}, kernel_volume={kg.kernel_volume}, ' \
               f'kernel_size={one(kg.kernel_size)}, stride={one(kg.kernel_stride)}, dilation={one(kg.kernel_dilation)}, ' \
               f'bn={self.bn is not None}, act={self.act_module.__class__.__name__.replace("Minkowski", "ME", 1)})'


class ConvBlock(BaseConvBlock):
    def __init__(self, in_channels, out_channels, kernel_size, stride, dilation=1, dimension=3,
                 region_type: str = 'HYPER_CUBE', bn: bool = False, bias: Optional[bool] = None,
                 act: Union[str, nn.Module, None] = 'relu'):
        super().__init__(ME.MinkowskiConvolution, in_channels, out_channels, kernel_size, stride, dilation, dimension,
                         region_type, bn, bias, act)


class ConvTransBlock(BaseConvBlock):
    def __init__(self, in_channels, out_channels, kernel_size, stride, dilation=1, dimension=3,
                 region_type: str = 'HYPER_CUBE', bn: bool = False, bias: Optional[bool] = None,
                 act: Union[str, nn.Module, None] = 'relu'):
        super().__init__(ME.MinkowskiConvolutionTranspose, in_channels, out_channels, kernel_size, stride, dilation,
                         dimension, region_type, bn, bias, act)


class GenConvTransBlock(BaseConvBlock):
    def __init__(self, in_channels, out_channels, kernel_size, stride, dilation=1, dimension=3,
                 region_type: str = 'HYPER_CUBE', bn: bool = False, bias: Optional[bool] = None,
                 act: Union[str, nn.Module, None] = 'relu'):
        super().__init__(ME.MinkowskiGenerativeConvolutionTranspose, in_channels, out_channels, kernel_size, stride,
                         dilation, dimension, region_type, bn, bias, act)


class ResBlock(nn.Module):
    """:162-190"""

    def __init__(self, channels, region_type: str, bn: bool, act: Optional[str], kernel_size: int = 3, last_act: bool = False):
        super().__init__()
        self.channels, self.bn, self.act, self.region_type, self.kernel_size = channels, bn, act, region_type, kernel_size
        self.last_act = get_act_module(act) if last_act is True else None
        self.conv0 = ConvBlock(channels, channels, kernel_size, 1, region_type=region_type, bn=bn, act=act)
        self.conv1 = ConvBlock(channels, channels, kernel_size, 1, region_type=region_type, bn=bn, act=None)

    def forward(self, x):
        out = self.conv1(self.conv0(x))
        out += x
        if self.last_act is not None:
            out = self.last_act(out)
        return out

    def __repr__(self):
        info = f'MEResBlock(channels={self.channels}, bn={self.bn}, act={self.act}'
        if self.kernel_size != 3:
            info += f', kernel_size={self.kernel_size}'
        if self.region_type != 'HYPER_CUBE':
            info += f', region_type={self.region_type}'
        return info + ')'


class InceptionResBlock(nn.Module):
    """:193-225"""

    def __init__(self, channels, region_type: str, bn: bool, act: Optional[str], kernel_size: int = 3):
        super().__init__()
        self.channels, self.bn, self.act, self.region_type, self.kernel_size = channels, bn, act, region_type, kernel_size
        self.path_0 = nn.Sequential(
            ConvBlock(channels, channels // 4, kernel_size, 1, region_type=region_type, bn=bn, act=act),
            ConvBlock(channels // 4, channels // 2, kernel_size, 1, region_type=region_type, bn=bn, act=None))
        self.path_1 = nn.Sequential(
            ConvBlock(channels, channels // 4, 1, 1, region_type=region_type, bn=bn, act=act),
            ConvBlock(channels // 4, channels // 4, kernel_size, 1, region_type=region_type, bn=bn, act=act),
            ConvBlock(channels // 4, channels // 2, 1, 1, region_type=region_type, bn=bn, act=None))

    def forward(self, x):
        return ME.cat(self.path_0(x), self.path_1(x)) + x

    def __repr__(self):
        info = f'MEInceptionResBlock(channels={self.channels}, bn={self.bn}, act={self.act}'
        if self.kernel_size != 3:
            info += f', kernel_size={self.kernel_size}'
        if self.region_type != 'HYPER_CUBE':
            info += f', region_type={self.region_type}'
        return info + ')'


class NNSequentialWithArgs(nn.Sequential):
    """:228-243: extra args go to the first block of `target_block_class`"""
    target_block_class = None

    def forward(self, x, *args, **kwargs):
        used_flag = False
        for m in self:
            if used_flag is False and isinstance(m, self.target_block_class):
                x = m(x, *args, **kwargs)
                used_flag = True
            else:
                x = m(x)
        if args or kwargs:
            assert used_flag
        return x


class NNSequentialWithConvTransBlockArgs(NNSequentialWithArgs):
    target_block_class = ConvTransBlock


class NNSequentialWithConvBlockArgs(NNSequentialWithArgs):
    target_block_class = ConvBlock


def minkowski_tensor_wrapped_op(x, operation: Callable[[torch.Tensor], Any], needs_recover: bool = True,
                                add_batch_dim: bool = False):
    """:252-280"""
    if needs_recover is True:
        assert add_batch_dim is False
    if isinstance(x, torch.Tensor):
        return operation(x)
    ret = operation(x.F)
    ret = list(ret) if isinstance(ret, Tuple) else [ret]
    for idx in range(len(ret)):
        if isinstance(ret[idx], torch.Tensor):
            if needs_recover is True:
                ret[idx] = ME.SparseTensor(features=ret[idx], coordinate_map_key=x.coordinate_map_key,
                                           coordinate_manager=x.coordinate_manager)
            elif add_batch_dim is True:
                ret[idx] = ret[idx][None]
    return ret[0] if len(ret) == 1 else tuple(ret)


def get_minkowski_tensor_coords_tuple(x):
    try:
        return x.coordinate_map_key, x.coordinate_manager
    except AttributeError:
        return None


def minkowski_tensor_split(x, split_size: Union[int, List[int]]) -> List:
    """:378-398"""
    if isinstance(split_size, list):
        ends = torch.cumsum(torch.tensor(split_size), dim=0).tolist()
        starts = [0] + ends[:-1]
    elif isinstance(split_size, int):
        n = math.ceil(x.F.shape[1] / split_size)
        assert n > 1
        starts = [i * split_size for i in range(n)]
        ends = starts[1:] + [x.F.shape[1]]
    else:
        raise NotImplementedError
    return [ME.SparseTensor(features=x.F[:, s:e], coordinate_map_key=x.coordinate_map_key,
                            coordinate_manager=x.coordinate_manager) for s, e in zip(starts, ends)]


def minkowski_expand_coord_2x(coord: torch.Tensor, current_tensor_stride: int):
    """:401-408"""
    assert coord.ndim == 2 and coord.shape[1] == 4
    strides = torch.tensor(((0, 0, 0, 0), (0, 1, 0, 0), (0, 0, 1, 0), (0, 1, 1, 0),
                            (0, 0, 0, 1), (0, 1, 0, 1), (0, 0, 1, 1), (0, 1, 1, 1)),
                           dtype=coord.dtype, device=coord.device) * (current_tensor_stride // 2)
    return coord.unsqueeze(1) + strides.unsqueeze(0)
