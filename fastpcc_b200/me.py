"""MinkowskiEngine-shaped shim over the B200 kernels: the subset of ME's public surface that the reference's
float layer API and lossy codecs touch (lib/minkowski_sparse_conv_layers.py:17-25,38-39,67-81,214,268-272;
lossy_coord_v2/layers.py:139-190; lossy_coord_lossy_color/geo_lossl_em.py:249-317).

ME itself (~0.5.4) is not vendored by the reference and cannot be installed offline; conventions follow its
published behaviour as pinned by the reference's call sites (see oracle/float_ops.py): absolute coordinates
(multiples of the tensor stride), HYPER_CUBE offsets with x fastest, odd kernels centred / even kernels 0..k-1,
kernel parameter [K, C_in, C_out] ([C_in, C_out] for 1x1), bias [1, C_out].

Differences that matter to a caller:
  * compute runs on tcgen05 tensor cores in fp16 (default) or bf16 with fp32 accumulation; parameters stay fp32 in
    the state dict, features travel in the compute dtype (`set_compute_dtype`);
  * coordinate sets are kept in Morton order (x least significant, ME's convention relied on at
    lossy_coord_v2/model.py:122-124), so generated / strided coordinates have a defined, reproducible row order;
  * a following activation can ride in the conv epilogue (`fused_act`), which is how ConvBlock uses it;
  * training: when grad is enabled and a parameter or the input features require it, every conv / linear layer runs
    through `autograd.MELayerFunction` -- the same forward kernels in the same order (the output bits do not depend on
    the grad mode), dgrad / wgrad on the tcgen05 kernels, the fused ReLU / LeakyReLU (slope >= 0) backward in one pass
    (`fpcc_act_grad_f16`).  On that path a PReLU or a negative LeakyReLU slope is applied after the layer as a torch op,
    so a PReLU slope trains.  Feature gradients travel in the compute dtype (fp32 for fp32 input features), parameter
    gradients are fp32.  Pruning, cat, +, batch norm and max (un)pooling are torch ops and differentiate as such: max
    pooling shares the gradient among tied maxima (torch's `scatter_reduce` amax rule), where ME routes it to one argmax.
"""
from enum import Enum
from typing import Dict, Optional, Tuple, Union

import torch
import torch.nn as nn

from . import ops

_COMPUTE = torch.float16


def set_compute_dtype(dtype):
    global _COMPUTE
    assert dtype in (torch.float16, torch.bfloat16)
    _COMPUTE = dtype


def compute_dtype():
    return _COMPUTE


class RegionType(Enum):
    HYPER_CUBE = 0


class SparseTensorOperationMode(Enum):
    SEPARATE_COORDINATE_MANAGER = 0
    SHARE_COORDINATE_MANAGER = 1


class MinkowskiAlgorithm(Enum):
    DEFAULT = 0
    MEMORY_EFFICIENT = 1
    SPEED_OPTIMIZED = 2


class CoordinateMapType(Enum):
    CPU = 0
    CUDA = 1


# ME's process-wide state (lossy_coord_v2/model.py:35,127-135,200-206): with SHARE_COORDINATE_MANAGER a SparseTensor
# built without an explicit manager joins the global one
_OPERATION_MODE = SparseTensorOperationMode.SEPARATE_COORDINATE_MANAGER
_GLOBAL_CM = None


def set_sparse_tensor_operation_mode(mode: SparseTensorOperationMode):
    global _OPERATION_MODE
    _OPERATION_MODE = mode


def sparse_tensor_operation_mode():
    return _OPERATION_MODE


def set_global_coordinate_manager(cm):
    global _GLOBAL_CM
    _GLOBAL_CM = cm


def global_coordinate_manager():
    return _GLOBAL_CM


def clear_global_coordinate_manager():
    global _GLOBAL_CM
    _GLOBAL_CM = None


def _publish(t: torch.Tensor):
    """a cached derived tensor may be read from another CUDA stream next: finish the kernels that fill it first"""
    if t.is_cuda:
        torch.cuda.current_stream(t.device).synchronize()


class SparseTensorQuantizationMode(Enum):
    RANDOM_SUBSAMPLE = 0
    UNWEIGHTED_AVERAGE = 1


def _triple(v):
    return tuple(int(x) for x in v) if isinstance(v, (tuple, list)) else (int(v),) * 3


class KernelGenerator:
    def __init__(self, kernel_size=-1, stride=1, dilation=1, region_type=RegionType.HYPER_CUBE, dimension=3, **_):
        assert region_type == RegionType.HYPER_CUBE, 'only HYPER_CUBE kernels are used by the reference configs'
        self.kernel_size, self.kernel_stride, self.kernel_dilation = _triple(kernel_size), _triple(stride), _triple(dilation)
        assert self.kernel_dilation == (1, 1, 1)
        self.region_type, self.dimension = region_type, dimension
        self.kernel_volume = self.kernel_size[0] * self.kernel_size[1] * self.kernel_size[2]


class CoordinateMapKey:
    def __init__(self, tensor_stride, tag=''):
        self.tensor_stride, self.tag = _triple(tensor_stride), tag

    def get_tensor_stride(self):
        return list(self.tensor_stride)

    def get_key(self):
        return (self.tensor_stride, self.tag)

    def __hash__(self):
        return hash(self.get_key())

    def __eq__(self, o):
        return isinstance(o, CoordinateMapKey) and self.get_key() == o.get_key()

    def __repr__(self):
        return f'CoordinateMapKey({self.tensor_stride}, {self.tag!r})'


def morton_order(coords: torch.Tensor, scale: int = 1) -> torch.Tensor:
    """argsort by (batch, Morton code with x least significant) of coords / scale"""
    c = coords if scale == 1 else torch.cat([coords[:, :1], coords[:, 1:] // scale], 1).contiguous()
    code = ops.morton_encode(c.contiguous(), col0=1, msb_axis=2)
    return torch.argsort(code + (c[:, 0].long() << 48) if int(c.shape[0]) else code)


class CoordinateManager:
    def __init__(self, D: int = 3, **_):
        self.D = D
        self._coords: Dict[CoordinateMapKey, torch.Tensor] = {}
        self._hash: Dict[CoordinateMapKey, Tuple[torch.Tensor, torch.Tensor]] = {}
        self._kmaps: Dict[tuple, torch.Tensor] = {}
        self._n_tags = 0
        self._manager = self  # ME exposes the C++ manager as `_manager` (lossy_coord_v2/layers.py:153)

    # -- coordinate sets ----------------------------------------------------------------------------------
    def _new_key(self, tensor_stride, coords, string_id: str = '') -> CoordinateMapKey:
        """ME names a coordinate map (tensor stride, string id): '' for inserted / strided maps, 'pruned' for the
        outputs of MinkowskiPruning and the maps derived from them; a taken name gets a numeric suffix."""
        key = CoordinateMapKey(tensor_stride, string_id)
        if key in self._coords:
            self._n_tags += 1
            key = CoordinateMapKey(tensor_stride, f'{string_id}#{self._n_tags}')
        self._coords[key] = coords.contiguous()
        return key

    def insert_and_map(self, coordinates: torch.Tensor, tensor_stride=1, string_id: str = ''):
        """Registers a coordinate set as given (the codecs pass unique, Morton-sorted coordinates,
        lossy_coord_v2/model.py:138-154).  Returns (key, (unique_index, inverse_index))."""
        assert coordinates.dtype == torch.int32 and coordinates.shape[1] == 4
        key = self._new_key(tensor_stride, coordinates, string_id)
        idx = torch.arange(coordinates.shape[0], device=coordinates.device)
        return key, (idx, idx)

    def get_coordinates(self, key: CoordinateMapKey) -> torch.Tensor:
        return self._coords[key]

    def hash_of(self, key):
        if key not in self._hash:
            self._hash[key] = ops.hash_build(self._coords[key], layout=0)
        return self._hash[key]

    def stride(self, in_key: CoordinateMapKey, stride) -> CoordinateMapKey:
        """Down-sampled coordinate set: unique(floor(c / (s*ts)) * (s*ts)), Morton ordered; cached per (key, stride)."""
        s = _triple(stride)
        tag = ('stride', in_key, s)
        if tag in self._kmaps:
            return self._kmaps[tag]
        ts = in_key.tensor_stride
        out_ts = tuple(a * b for a, b in zip(ts, s))
        c = self._coords[in_key].clone()
        for a in range(3):
            c[:, a + 1] = torch.div(c[:, a + 1], out_ts[a], rounding_mode='floor') * out_ts[a]
        c = c[morton_order(c, out_ts[0])]
        c = torch.unique_consecutive(c, dim=0)
        key = self._new_key(out_ts, c, in_key.tag.split('#')[0])
        self._kmaps[tag] = key
        return key

    def origin_map(self, key: CoordinateMapKey):
        """ME: (origin key, list of row-index tensors, one per batch sample) of the global (origin) pooling map."""
        tag = ('origin', key)
        if tag not in self._kmaps:
            b = self._coords[key][:, 0].long()
            n_batch = int(b.max().item()) + 1 if b.numel() else 0
            order = torch.argsort(b, stable=True)
            counts = torch.bincount(b, minlength=n_batch).tolist()
            self._kmaps[tag] = list(torch.split(order, counts))
        return CoordinateMapKey(tuple(0 for _ in key.tensor_stride), 'origin'), self._kmaps[tag]

    def get_coordinate_map_keys(self, tensor_stride):
        ts = _triple(tensor_stride)
        return [k for k in self._coords if tuple(k.tensor_stride) == ts]

    def parent_rows(self, in_key: CoordinateMapKey, out_key: CoordinateMapKey) -> torch.Tensor:
        """row of `out_key` (coarser) that contains each voxel of `in_key`, -1 if absent; cached"""
        tag = ('parent', in_key, out_key)
        if tag not in self._kmaps:
            ots = torch.tensor(out_key.tensor_stride, device=self._coords[in_key].device, dtype=torch.int32)
            par = self._coords[in_key].clone()
            par[:, 1:] = torch.div(par[:, 1:], ots, rounding_mode='floor') * ots
            keys, vals = self.hash_of(out_key)
            self._kmaps[tag] = (ops.kmap_lookup(keys, vals, par.contiguous(), (1, 1, 1), (1, 1, 1), convention=1)[0] - 1).long()
        return self._kmaps[tag]

    def kernel_table(self, in_key, out_key, kernel_size, scale) -> torch.Tensor:
        """k-major neighbour table [K, N_out] (input row + 1 | 0), ME offset convention, cached."""
        tag = ('kmap', in_key, out_key, _triple(kernel_size), _triple(scale))
        if tag not in self._kmaps:
            keys, vals = self.hash_of(in_key)
            self._kmaps[tag] = ops.kmap_lookup(keys, vals, self._coords[out_key], _triple(kernel_size), _triple(scale), convention=1)
        return self._kmaps[tag]

    def grouped_kernel_table(self, in_key, out_key, kernel_size, scale):
        """(table with its columns regrouped by neighbour pattern, row permutation) for the conv kernel, cached;
        skipped (all-empty) offsets contribute exact zeros, so the fp32 sums are bit-identical to the plain table's."""
        tag = ('kmap_grouped', in_key, out_key, _triple(kernel_size), _triple(scale))
        if tag not in self._kmaps:
            self._kmaps[tag] = ops.group_rows(self.kernel_table(in_key, out_key, kernel_size, scale))
        return self._kmaps[tag]

    def kernel_map(self, in_key, out_key, stride=1, kernel_size=3, region_type=None, **_):
        """ME's dict {kernel index: [2, n] (in rows, out rows)} (used with kernel_size=1 by get_coord_mask,
        geo_lossl_em.py:306-317)."""
        table = self.kernel_table(in_key, out_key, kernel_size, in_key.tensor_stride)
        in_map, out_map, offsets = ops.kmap_compact(table)
        off = offsets.tolist()
        return {k: torch.stack([in_map[off[k]: off[k + 1]], out_map[off[k]: off[k + 1]]]).long()
                for k in range(table.shape[0]) if off[k + 1] > off[k]}


GROUP_ROWS_MIN = 4096  # below this a conv is launch-bound and sorting the rows does not pay


class SparseTensor:
    def __init__(self, features: torch.Tensor, coordinates: Optional[torch.Tensor] = None, tensor_stride=1,
                 coordinate_map_key: Optional[CoordinateMapKey] = None, coordinate_manager: Optional[CoordinateManager] = None,
                 quantization_mode=None, device=None, **_):
        if coordinate_manager is None and coordinate_map_key is None and _OPERATION_MODE == SparseTensorOperationMode.SHARE_COORDINATE_MANAGER:
            if _GLOBAL_CM is None:
                set_global_coordinate_manager(CoordinateManager())
            coordinate_manager = _GLOBAL_CM
        if coordinate_manager is None:
            coordinate_manager = CoordinateManager()
        if coordinate_map_key is None:
            assert coordinates is not None
            if device is not None:
                coordinates, features = coordinates.to(device), features.to(device)
            coordinate_map_key, _ = coordinate_manager.insert_and_map(coordinates.to(torch.int32).contiguous(), tensor_stride)
        self._F = features
        self.coordinate_map_key, self.coordinate_manager = coordinate_map_key, coordinate_manager

    @property
    def F(self):
        return self._F

    @property
    def C(self):
        return self.coordinate_manager.get_coordinates(self.coordinate_map_key)

    @property
    def tensor_stride(self):
        return list(self.coordinate_map_key.tensor_stride)

    @property
    def shape(self):
        return self._F.shape

    @property
    def device(self):
        return self._F.device

    @property
    def dtype(self):
        return self._F.dtype

    def _like(self, f):
        return SparseTensor(f, coordinate_map_key=self.coordinate_map_key, coordinate_manager=self.coordinate_manager)

    # -- per-sample views (ME: SparseTensor.decomposition_permutations / decomposed_coordinates / decomposed_features)
    @property
    def _batchwise_row_indices(self):
        return self.coordinate_manager.origin_map(self.coordinate_map_key)[1]

    @property
    def decomposition_permutations(self):
        return self._batchwise_row_indices

    @property
    def decomposed_coordinates(self):
        c = self.C
        return [c[rows, 1:] for rows in self._batchwise_row_indices]

    @property
    def decomposed_features(self):
        return [self._F[rows] for rows in self._batchwise_row_indices]

    @property
    def decomposed_coordinates_and_features(self):
        return self.decomposed_coordinates, self.decomposed_features

    def __add__(self, o):
        if isinstance(o, SparseTensor):
            assert o.coordinate_map_key == self.coordinate_map_key, 'addition needs identical coordinate sets'
            return self._like(self._F + o._F)
        return self._like(self._F + o)

    __iadd__ = __add__

    def __repr__(self):
        return f'SparseTensor(F={tuple(self._F.shape)} {self._F.dtype}, stride={self.tensor_stride})'


def cat(*tensors):
    tensors = tensors[0] if len(tensors) == 1 and isinstance(tensors[0], (list, tuple)) else tensors
    assert all(t.coordinate_map_key == tensors[0].coordinate_map_key for t in tensors)
    return tensors[0]._like(torch.cat([t.F for t in tensors], 1))


# ------------------------------------------------------------------------------------------------------------
# modules
# ------------------------------------------------------------------------------------------------------------
_ACT = {'none': (ops.ACT_NONE, 0.0), 'relu': (ops.ACT_RELU, 0.0)}


def _fusable_act(act) -> bool:
    """an activation module (or None) that the conv / linear epilogue can apply"""
    return act is None or isinstance(act, (MinkowskiReLU, MinkowskiLeakyReLU)) or (isinstance(act, MinkowskiPReLU) and act.weight.numel() == 1)


def _act_code(act) -> Tuple[int, float]:
    """(code, slope) of a fusable activation module / None"""
    if act is None:
        return ops.ACT_NONE, 0.0
    if isinstance(act, MinkowskiReLU):
        return ops.ACT_RELU, 0.0
    if isinstance(act, MinkowskiLeakyReLU):
        return ops.ACT_LEAKY, float(act.negative_slope)
    if isinstance(act, MinkowskiPReLU) and act.weight.numel() == 1:
        return ops.ACT_LEAKY, float(act.weight.item())
    return -1, 0.0


def _needs_grad(f: torch.Tensor, *params) -> bool:
    return torch.is_grad_enabled() and (f.requires_grad or any(p is not None and p.requires_grad for p in params))


def _epilogue_act(act, grad: bool):
    """-> (code, slope, module applied after the layer | None).  Inference fuses every fusable activation.  With grad the
    epilogue keeps only activations whose derivative follows from the output (ReLU, LeakyReLU with slope >= 0); a PReLU
    (its slope may train; no host read of it) and a negative LeakyReLU slope run after the layer as torch ops."""
    if grad and (isinstance(act, MinkowskiPReLU) or (isinstance(act, MinkowskiLeakyReLU) and act.negative_slope < 0)):
        return ops.ACT_NONE, 0.0, act
    code, slope = _act_code(act)
    return code, slope, None


def _differentiable(x, kernel, bias, c_in, c_out, code, slope, run, after, out_key, kind, **spec):
    """the output SparseTensor of a conv / linear layer on the training path: `run()` is the layer's inference call"""
    from . import autograd  # imported here: oracle/me_cpu.py executes this file's source outside the package
    sp = autograd.MESpec(kind, c_in, c_out, code, slope, _COMPUTE, **spec)
    out = SparseTensor(autograd.me_layer(x.F, kernel, bias, sp, run), coordinate_map_key=out_key, coordinate_manager=x.coordinate_manager)
    return after(out) if after is not None else out


def _as_compute(f: torch.Tensor) -> torch.Tensor:
    return f if f.dtype == _COMPUTE else f.to(_COMPUTE)


class _ConvBase(nn.Module):
    def __init__(self, in_channels, out_channels, kernel_size=-1, stride=1, dilation=1, bias=False,
                 kernel_generator: Optional[KernelGenerator] = None, dimension=3, **_):
        super().__init__()
        if kernel_generator is None:
            kernel_generator = KernelGenerator(kernel_size, stride, dilation, dimension=dimension)
        self.kernel_generator = kernel_generator
        self.in_channels, self.out_channels, self.dimension = in_channels, out_channels, dimension
        kv = kernel_generator.kernel_volume
        shape = (kv, in_channels, out_channels) if kv > 1 else (in_channels, out_channels)
        self.kernel = nn.Parameter(torch.empty(shape))
        self.bias = nn.Parameter(torch.zeros(1, out_channels)) if bias else None
        with torch.no_grad():
            n = in_channels * kv
            self.kernel.uniform_(-(1.0 / n) ** 0.5, (1.0 / n) ** 0.5)
        self._cache = None

    def _weights(self):
        """([K, C_out_pad, C_in_pad] compute-dtype weight for the kernels, fp32 bias [C_out_pad] | None)"""
        key = (self.kernel._version, self.kernel.data_ptr(), _COMPUTE, None if self.bias is None else self.bias._version)
        if self._cache is None or self._cache[0] != key:
            k = self.kernel.detach()
            w = ops.f16_weight(k[None] if k.dim() == 2 else k, _COMPUTE)
            cout_p, cin_p = w.shape[1:]
            b = None
            if self.bias is not None:
                b = torch.zeros(cout_p, dtype=torch.float32, device=k.device)
                b[:k.shape[-1]] = self.bias.detach().reshape(-1).float()
            _publish(w)
            self._cache = (key, w, b, cin_p, cout_p)
        return self._cache[1:]

    def _run(self, f, table, act, slope, residual=None, row_perm=None):
        w, b, cin_p, cout_p = self._weights()
        f = ops.pad_cols(_as_compute(f), cin_p).contiguous()
        if residual is not None:
            residual = ops.pad_cols(_as_compute(residual), cout_p).contiguous()
        kv = w.shape[0]
        # single-channel heads (occupancy logits, top-k scores, the clipped bottom feature) keep the fp32 accumulator:
        # rounded to fp16 they collide into ties that the codecs' `kthvalue` / `>` selections (lossy_coord_v2/layers.py:
        # 166-176) and 16-bit probabilities (geo_lossl_em.py:95-99) would see
        od = torch.float32 if (self.out_channels == 1 and residual is None) else None
        if kv == 1:
            out = ops.linear_f16(f, w[0], bias=b, act=act, slope=slope, residual=residual, out_dtype=od)
        else:
            out = ops.spconv_f16(f, w, table, bias=b, act=act, slope=slope, residual=residual, row_perm=row_perm, out_dtype=od)
        return out[:, :self.out_channels] if cout_p != self.out_channels else out


class MinkowskiConvolution(_ConvBase):
    def forward(self, x: SparseTensor, coordinates: Optional[CoordinateMapKey] = None, fused_act=None) -> SparseTensor:
        cm, kg = x.coordinate_manager, self.kernel_generator
        grad = _needs_grad(x.F, self.kernel, self.bias)
        code, slope, after = _epilogue_act(fused_act, grad)
        assert code >= 0, 'activation cannot be fused'
        if kg.kernel_stride == (1, 1, 1):
            out_key = x.coordinate_map_key if coordinates is None else coordinates
        else:
            out_key = cm.stride(x.coordinate_map_key, kg.kernel_stride) if coordinates is None else coordinates
        table = perm = None
        if kg.kernel_volume > 1:
            args = (x.coordinate_map_key, out_key, kg.kernel_size, x.coordinate_map_key.tensor_stride)
            if cm.get_coordinates(out_key).shape[0] >= GROUP_ROWS_MIN:
                table, perm = cm.grouped_kernel_table(*args)
            else:
                table = cm.kernel_table(*args)
        if grad:
            kv = kg.kernel_volume
            return _differentiable(x, self.kernel, self.bias, self.in_channels, self.out_channels, code, slope,
                                   lambda: self._run(x.F, table, code, slope, row_perm=perm), after, out_key,
                                   'conv' if kv > 1 else 'linear', layout='kio' if kv > 1 else 'io',
                                   table=cm.kernel_table(*args) if kv > 1 else None, group=x.F.shape[0] >= GROUP_ROWS_MIN)
        f = self._run(x.F, table, code, slope, row_perm=perm)
        return SparseTensor(f, coordinate_map_key=out_key, coordinate_manager=cm)


class MinkowskiConvolutionTranspose(_ConvBase):
    """kernel = stride = 2 onto an EXISTING finer coordinate set (`coordinates` key): every output voxel has exactly
    one parent, so the layer is one weight block per child slot (the selection form of the linear kernel)."""

    def forward(self, x: SparseTensor, coordinates: CoordinateMapKey, fused_act=None) -> SparseTensor:
        cm, kg = x.coordinate_manager, self.kernel_generator
        assert kg.kernel_size == (2, 2, 2) and kg.kernel_stride == (2, 2, 2), 'only k=2, s=2 transposed convs are used'
        grad = _needs_grad(x.F, self.kernel, self.bias)
        code, slope, after = _epilogue_act(fused_act, grad)
        ts = x.coordinate_map_key.tensor_stride[0]
        half = ts // 2
        oc = cm.get_coordinates(coordinates)
        tag = ('tconv', x.coordinate_map_key, coordinates)
        if tag not in cm._kmaps:
            parent = oc.clone()
            parent[:, 1:] = torch.div(oc[:, 1:], ts, rounding_mode='floor') * ts
            keys, vals = cm.hash_of(x.coordinate_map_key)
            par = ops.kmap_lookup(keys, vals, parent.contiguous(), (1, 1, 1), (1, 1, 1), convention=1)[0] - 1  # -1: no parent
            d = (oc[:, 1:] - parent[:, 1:]) // half
            slot = (d[:, 0] + 2 * d[:, 1] + 4 * d[:, 2]).to(torch.uint8)  # x fastest
            slot = torch.where(par >= 0, slot, torch.full_like(slot, 255))  # orphans join no group -> bias only
            cm._kmaps[tag] = ops.slot_pairs(par.clamp(min=0).contiguous(), slot.contiguous())
            cm._kmaps[('tconv_slots',) + tag[1:]] = (par.clamp(min=0).contiguous(), slot.contiguous())
        sel = cm._kmaps[tag]

        def run():
            w, b, cin_p, cout_p = self._weights()
            f = ops.pad_cols(_as_compute(x.F), cin_p).contiguous()
            # rows without a parent belong to no group: they keep act(bias)
            fill = torch.zeros(cout_p, dtype=torch.float32, device=f.device) if b is None else b
            fill = torch.relu(fill) if code == ops.ACT_RELU else (torch.where(fill < 0, fill * slope, fill) if code == ops.ACT_LEAKY else fill)
            out = fill.to(_COMPUTE)[None].repeat(oc.shape[0], 1)
            res = ops.linear_f16(f, w.reshape(8 * cout_p, cin_p), bias=b, act=code, slope=slope, sel=sel, n_out_rows=oc.shape[0], out=out)
            return res[:, :self.out_channels] if cout_p != self.out_channels else res

        if grad:
            ttag = ('tconv_table',) + tag[1:]
            if ttag not in cm._kmaps:  # k-major [8, n_child]: parent row + 1 in the child's slot row (the conv form of sel)
                cm._kmaps[ttag] = ops.slot_table(*cm._kmaps[('tconv_slots',) + tag[1:]])
            return _differentiable(x, self.kernel, self.bias, self.in_channels, self.out_channels, code, slope, run, after,
                                   coordinates, 'tconv', table=cm._kmaps[ttag], group=x.F.shape[0] >= GROUP_ROWS_MIN)
        return SparseTensor(run(), coordinate_map_key=coordinates, coordinate_manager=cm)


class MinkowskiGenerativeConvolutionTranspose(_ConvBase):
    """kernel = stride = 2: generates all 8 children of every input voxel (rows ordered parent-major, child x fastest,
    i.e. Morton order when the input is Morton ordered); one dense linear C_in -> 8*C_out."""

    def forward(self, x: SparseTensor, coordinates=None, fused_act=None) -> SparseTensor:
        cm, kg = x.coordinate_manager, self.kernel_generator
        assert kg.kernel_size == (2, 2, 2) and kg.kernel_stride == (2, 2, 2), 'only k=2, s=2 generative convs are used'
        grad = _needs_grad(x.F, self.kernel, self.bias)
        code, slope, after = _epilogue_act(fused_act, grad)
        ts = x.coordinate_map_key.tensor_stride[0]
        half = ts // 2
        tag = ('gen', x.coordinate_map_key)
        if tag not in cm._kmaps:
            c = x.C
            offs = torch.tensor([[0, k & 1, (k >> 1) & 1, (k >> 2) & 1] for k in range(8)], dtype=torch.int32, device=c.device) * half
            cm._kmaps[tag] = cm._new_key((half,) * 3, (c[:, None] + offs[None]).reshape(-1, 4))
        out_key = cm._kmaps[tag]

        def run():
            w, b, cin_p, cout_p = self._weights()
            f = ops.pad_cols(_as_compute(x.F), cin_p).contiguous()
            b8 = None if b is None else b.repeat(8)
            res = ops.linear_f16(f, w.reshape(8 * cout_p, cin_p), bias=b8, act=code, slope=slope)
            res = res.reshape(-1, cout_p)
            return res[:, :self.out_channels] if cout_p != self.out_channels else res

        if grad:
            return _differentiable(x, self.kernel, self.bias, self.in_channels, self.out_channels, code, slope, run, after,
                                   out_key, 'gen')
        return SparseTensor(run(), coordinate_map_key=out_key, coordinate_manager=cm)


class MinkowskiLinear(nn.Module):
    def __init__(self, in_features, out_features, bias=True):
        super().__init__()
        self.linear = nn.Linear(in_features, out_features, bias=bias)
        self._cache = None

    def forward(self, x: SparseTensor, fused_act=None) -> SparseTensor:
        lin = self.linear
        grad = _needs_grad(x.F, lin.weight, lin.bias)
        code, slope, after = _epilogue_act(fused_act, grad)
        key = (lin.weight._version, lin.weight.data_ptr(), _COMPUTE, None if lin.bias is None else lin.bias._version)
        if self._cache is None or self._cache[0] != key:
            w = ops.f16_weight(lin.weight.t()[None], _COMPUTE)[0]
            cout_p, cin_p = w.shape
            b = None
            if lin.bias is not None:
                b = torch.zeros(cout_p, dtype=torch.float32, device=w.device)
                b[:lin.out_features] = lin.bias.detach().float()
            _publish(w)
            self._cache = (key, w, b, cin_p, cout_p)
        _, w, b, cin_p, cout_p = self._cache

        def run():
            f = ops.pad_cols(_as_compute(x.F), cin_p).contiguous()
            od = torch.float32 if lin.out_features == 1 else None  # single-channel heads keep fp32 (see _ConvBase._run)
            out = ops.linear_f16(f, w, bias=b, act=code, slope=slope, out_dtype=od)
            return out[:, :lin.out_features] if cout_p != lin.out_features else out

        if grad:
            return _differentiable(x, lin.weight, lin.bias, lin.in_features, lin.out_features, code, slope, run, after,
                                   x.coordinate_map_key, 'linear', layout='oi')
        return x._like(run())


class _Pointwise(nn.Module):
    def forward(self, x: SparseTensor) -> SparseTensor:
        return x._like(self.fn(x.F))


class MinkowskiReLU(_Pointwise):
    def __init__(self, inplace=False):
        super().__init__()

    def fn(self, f):
        return torch.relu(f)


class MinkowskiLeakyReLU(_Pointwise):
    def __init__(self, negative_slope=0.01, inplace=False):
        super().__init__()
        self.negative_slope = negative_slope

    def fn(self, f):
        return torch.nn.functional.leaky_relu(f, self.negative_slope)


class MinkowskiPReLU(_Pointwise):
    def __init__(self, num_parameters=1, init=0.25):
        super().__init__()
        self.weight = nn.Parameter(torch.full((num_parameters,), float(init)))

    def fn(self, f):
        return torch.nn.functional.prelu(f, self.weight.to(f.dtype))


class MinkowskiSigmoid(_Pointwise):
    def fn(self, f):
        return torch.sigmoid(f)


class MinkowskiBatchNorm(nn.Module):
    def __init__(self, num_features, **kw):
        super().__init__()
        self.bn = nn.BatchNorm1d(num_features, **kw)

    def forward(self, x: SparseTensor) -> SparseTensor:
        return x._like(self.bn(x.F.float()).to(x.F.dtype))


class MinkowskiMaxPooling(nn.Module):
    """kernel_size == stride (non-overlapping cells), as used by the top-k pruning (lossy_coord_v2/layers.py:159):
    max of the features of every coarse cell.  forward(x, coordinates=key) pools onto an existing coarser key."""

    def __init__(self, kernel_size, stride=1, dilation=1, kernel_generator=None, dimension=3):
        super().__init__()
        self.kernel_size, self.stride = _triple(kernel_size), _triple(stride)
        assert self.kernel_size == self.stride, 'only non-overlapping pooling (kernel_size == stride) is used by the codecs'

    def forward(self, x: SparseTensor, coordinates: Optional[CoordinateMapKey] = None) -> SparseTensor:
        cm = x.coordinate_manager
        out_key = cm.stride(x.coordinate_map_key, self.stride) if coordinates is None else coordinates
        par = cm.parent_rows(x.coordinate_map_key, out_key)
        assert bool((par >= 0).all()), 'max pooling: a voxel has no cell in the target coordinate set'
        n_out = cm.get_coordinates(out_key).shape[0]
        f = x.F
        out = torch.full((n_out, f.shape[1]), float('-inf'), dtype=f.dtype, device=f.device)
        out.scatter_reduce_(0, par[:, None].expand(-1, f.shape[1]), f, reduce='amax')
        return SparseTensor(out, coordinate_map_key=out_key, coordinate_manager=cm)


class MinkowskiPoolingTranspose(nn.Module):
    """kernel_size == stride un-pooling onto an existing finer key: every fine voxel receives its cell's feature."""

    def __init__(self, kernel_size, stride, dilation=1, kernel_generator=None, expand_coordinates=False, dimension=3):
        super().__init__()
        self.kernel_size, self.stride = _triple(kernel_size), _triple(stride)
        assert self.kernel_size == self.stride

    def forward(self, x: SparseTensor, coordinates: CoordinateMapKey) -> SparseTensor:
        cm = x.coordinate_manager
        par = cm.parent_rows(coordinates, x.coordinate_map_key)
        f = x.F[par.clamp(min=0)]
        f = torch.where((par >= 0)[:, None], f, torch.zeros_like(f))
        return SparseTensor(f, coordinate_map_key=coordinates, coordinate_manager=cm)


class MinkowskiPruning(nn.Module):
    def forward(self, x: SparseTensor, mask: torch.Tensor) -> SparseTensor:
        assert mask.dtype == torch.bool and mask.shape[0] == x.F.shape[0]
        cm = x.coordinate_manager
        key = cm._new_key(x.coordinate_map_key.tensor_stride, x.C[mask], 'pruned')
        return SparseTensor(x.F[mask], coordinate_map_key=key, coordinate_manager=cm)
