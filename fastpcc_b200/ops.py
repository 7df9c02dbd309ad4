"""Thin torch-tensor front-end over the C ABI (include/fastpcc_b200.h).

PyTorch is plumbing here: device memory, the current CUDA stream, and a few index/concat ops.  Every
computation on the hot path is a kernel of libfastpcc_b200.so; nothing falls back to torch or the CPU.
"""
import ctypes as C
import threading

import torch

from . import _lib
from ._lib import Epilogue

OUT_I8, OUT_I16, OUT_I32 = 0, 1, 2
_OUT_DTYPE = {OUT_I8: torch.int8, OUT_I16: torch.int16, OUT_I32: torch.int32}
CDF_LD = 256  # row pitch (entries) of device-resident CDF tables -> 16-byte loads in the decoder


def _s():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


def _need(t, dtype, name, dim=None):
    if t.dtype != dtype:
        raise RuntimeError(f'{name}: expected {dtype}, got {t.dtype}')
    if not t.is_cuda:
        raise RuntimeError(f'{name}: expected a CUDA tensor')
    if not t.is_contiguous():
        raise RuntimeError(f'{name}: expected a contiguous tensor')
    if dim is not None and t.dim() != dim:
        raise RuntimeError(f'{name}: expected {dim} dims, got {t.dim()}')
    return t


# ---- optional per-launch profiling (bench.py's instrumented pass; off on the timed path) -------------
_prof = None


def enable_profile(on: bool):
    """When on, every C-ABI call is bracketed by CUDA events on the current stream."""
    global _prof
    _prof = [] if on else None
    _pairs_cache.clear()  # its entries keep kernel maps alive: only for the duration of one instrumented pass
    return _prof


def _call(name, *args, tag=None, work=None):
    if _prof is None:
        return _lib.call(name, *args)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    _lib.call(name, *args)
    e1.record()
    _prof.append((tag or name, e0, e1, work or {}))


def profile_summary(prof):
    torch.cuda.synchronize()
    out = {}
    for tag, e0, e1, work in prof:
        d = out.setdefault(tag, {'ms': 0.0, 'launches': 0, 'ops': 0.0, 'mma_ops': 0.0, 'bytes': 0.0})
        d['ms'] += e0.elapsed_time(e1)
        d['launches'] += 1
        for k, v in work.items():
            if not isinstance(v, str):
                d[k] = d.get(k, 0.0) + v
    return out


def mma_i8_peak(iters=20000, n=256):
    """measured kind::i8 tensor-pipe ceiling of the current GPU in TOP/s (synchronises)"""
    out = C.c_double(0.0)
    _lib.call('fpcc_mma_i8_peak', int(iters), int(n), C.byref(out), _s())
    return out.value


def gemm_engine(k, n, kvol=1, zp_comp=False):
    """'tc' when the C side routes this shape to the tcgen05 kernel, else 'simt'."""
    return 'tc' if _lib.load().fpcc_gemm_engine(int(k), int(n), int(kvol), int(bool(zp_comp))) == 1 else 'simt'


_pairs_cache = {}


def _pairs_of(table):
    """matched pairs of a kernel map (instrumented pass only).  The entry holds the table itself, so its address cannot be
    reused by another map while the count is cached (a bare data_ptr key could hand back a stale count)."""
    key = (table.data_ptr(), tuple(table.shape), table._version)
    ent = _pairs_cache.get(key)
    if ent is None:
        if len(_pairs_cache) > 64:
            _pairs_cache.clear()
        ent = (table, int(torch.count_nonzero(table).item()))
        _pairs_cache[key] = ent
    return ent[1]


_ws_cache = {}


def workspace(nbytes, device):
    """Grow-only scratch buffer per (device, stream): kernels on one stream run in order, so reuse is safe."""
    key = (device.index if device.index is not None else torch.cuda.current_device(), _s())
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=device)
        _ws_cache[key] = buf
    return buf


def _ep_out_dtype(ep):
    """dtype of the rows a fused kernel writes to `out`: int8 when the second stage replaces the int32 rows (no aux_out)"""
    return torch.int8 if (ep.post_requant_mul and not ep.aux_out) else _OUT_DTYPE[ep.out_type]


def make_epilogue(requant_mul, zero_point, shift, out_type, bias=None, slope=None, residual=None, post_slope=None,
                  row_bias=None, post_requant=None, aux_out=None):
    """post_requant = (mul uint32[1], zero_point int64[1], shift, slope int32[1] | None): the fused second stage of the
    tensor-core kernels -- an int32 (Q8.23) result is not stored, the consumer's [PReLUIn32Out32 +] RequantFxpToScaledInt8
    runs in the same epilogue and int8 rows come out (fpcc_epilogue::post_requant_mul).  With `aux_out` (int8 [rows, ch])
    the int32 rows are ALSO stored (dual output for int32 tensors with a second consumer)."""
    _need(requant_mul, torch.uint32, 'requant_mul')
    _need(zero_point, torch.int64, 'zero_point')
    if shift < 0:
        raise RuntimeError(f'right shift must be >= 0, got {shift}')
    e = Epilogue()
    e.bias = _p(_need(bias, torch.int32, 'bias')) if bias is not None else None
    e.slope = _p(_need(slope, torch.int32, 'slope')) if slope is not None else None
    e.requant_mul = _p(requant_mul)
    e.zero_point = _p(zero_point)
    e.shift = int(shift)
    e.out_type = out_type
    e.mul_is_scalar = 1 if requant_mul.numel() == 1 else 0
    e.residual = _p(_need(residual, torch.int32, 'residual')) if residual is not None else None
    e.post_slope = _p(_need(post_slope, torch.int32, 'post_slope')) if post_slope is not None else None
    if row_bias is not None:
        table, idx = row_bias[:2]
        e.row_bias = _p(_need(table, torch.int32, 'row_bias table', 2))
        e.row_idx = _p(_need(idx, torch.uint8, 'row_bias index', 1))
        e.row_bias_bound = int(row_bias[2]) if len(row_bias) > 2 else 0  # max |table entry| when the caller knows it
    if post_requant is not None:
        mul2, zp2, shift2, slope2 = post_requant
        if out_type != OUT_I32:
            raise RuntimeError('post_requant needs an int32 first stage')
        e.post_requant_mul = _p(_need(mul2, torch.uint32, 'post requant_mul'))
        e.post_zero_point = _p(_need(zp2, torch.int64, 'post zero_point'))
        e.post_shift = int(shift2)
        e.post_requant_slope = _p(_need(slope2, torch.int32, 'post slope')) if slope2 is not None else None
    if aux_out is not None:
        # dual output: the int32 rows go to `out` as usual, the second stage's int8 rows to aux_out [rows, ch]
        if post_requant is None:
            raise RuntimeError('aux_out needs post_requant (the second stage whose int8 rows it receives)')
        e.aux_out = _p(_need(aux_out, torch.int8, 'aux_out', 2))
    e._keep = (bias, slope, requant_mul, zero_point, residual, post_slope, row_bias, post_requant, aux_out)
    return e


# Derived tensors that are cached and then read by every thread / CUDA stream (concurrent coding groups) follow ONE
# rule: they are created under `cache_lock` by exactly one thread, their producing stream is synchronised BEFORE the
# cache entry becomes visible, and a valid entry is never replaced.  (Replacing an entry frees a tensor that another
# stream's pending kernels may still read: the caching allocator only orders reuse on the allocating stream.)
cache_lock = threading.RLock()


def publish_ready(device=None):
    torch.cuda.current_stream(device).synchronize()


_identity = {}


def identity_epilogue(device):
    """acc*1 + 0 >> 0 -> int32: returns the raw accumulator (sparse_conv_in8w8out32's contract)."""
    key = device.index if device.index is not None else torch.cuda.current_device()
    ent = _identity.get(key)
    if ent is None:
        with cache_lock:
            ent = _identity.get(key)
            if ent is None:
                ent = (torch.ones(1, dtype=torch.int32).view(torch.uint32).to(device), torch.zeros(1, dtype=torch.int64, device=device))
                publish_ready(device)
                _identity[key] = ent
    mul, zp = ent
    return make_epilogue(mul, zp, 0, OUT_I32)


# ---------------------------------------------------------------------------------------------
# coordinates / kernel maps
# ---------------------------------------------------------------------------------------------

def hash_build(coords, layout=0, keys=None, vals=None):
    _need(coords, torch.int32, 'coords', 2)
    n = coords.shape[0]
    if keys is None:
        keys = torch.zeros(2 * n + 2, dtype=torch.int64, device=coords.device)
        vals = torch.zeros(2 * n + 2, dtype=torch.int32, device=coords.device)
    _call('fpcc_hash_insert_coords', _p(keys), _p(vals), keys.numel(), _p(coords), n, layout, _s(),
          work={'bytes': 28.0 * n})  # 16 B coords + 12 B table entry per point
    return keys, vals


def kmap_lookup(keys, vals, out_coords, kernel_size, stride, layout=0, k_major=True, pad_rows=None, convention=0):
    _need(out_coords, torch.int32, 'out_coords', 2)
    n = out_coords.shape[0]
    kv = kernel_size[0] * kernel_size[1] * kernel_size[2]
    if k_major:
        table = torch.empty((kv, n), dtype=torch.int32, device=out_coords.device)
        ld = n
    else:
        rows = n if pad_rows is None else pad_rows
        table = (torch.zeros if rows != n else torch.empty)((rows, kv), dtype=torch.int32, device=out_coords.device)
        ld = 0
    _call('fpcc_kmap_lookup', _p(keys), _p(vals), keys.numel(), _p(out_coords), n, layout,
              kernel_size[0], kernel_size[1], kernel_size[2], stride[0], stride[1], stride[2], convention,
              _p(table), 1 if k_major else 0, ld, _s(),
          work={'bytes': 16.0 * n + 12.0 * kv * n})  # coords + one 8-byte key probe and a 4-byte entry per (offset, row)
    return table


def kmap_compact(table, omit_k=-1):
    """k-major table -> (in_map, out_map, offsets[kvol+1]) on the device, no host sync."""
    kv, n = table.shape
    dev = table.device
    in_map = torch.empty(kv * n, dtype=torch.int32, device=dev)
    out_map = torch.empty(kv * n, dtype=torch.int32, device=dev)
    offsets = torch.empty(kv + 1, dtype=torch.int32, device=dev)
    nb = _lib.load().fpcc_kmap_compact_workspace(kv, n)
    ws = workspace(nb, dev)
    _call('fpcc_kmap_compact', _p(table), kv, n, n, omit_k, _p(in_map), _p(out_map), _p(offsets), _p(ws), ws.numel(), _s())
    return in_map, out_map, offsets


def downsample(coords, want_parent=True):
    """-> (parent_coords[n], occ[n], parent_of_child[n], slot_of_child[n], n_out_dev[1]); rows beyond n_out are junk."""
    _need(coords, torch.int32, 'coords', 2)
    n, dev = coords.shape[0], coords.device
    out_c = torch.empty((n, 4), dtype=torch.int32, device=dev)
    occ = torch.empty(n, dtype=torch.uint8, device=dev)
    par = torch.empty(n, dtype=torch.int32, device=dev) if want_parent else None
    slot = torch.empty(n, dtype=torch.uint8, device=dev) if want_parent else None
    cnt = torch.empty(1, dtype=torch.int32, device=dev)
    ws = workspace(_lib.load().fpcc_scan_workspace(n), dev)
    _call('fpcc_downsample', _p(coords), n, _p(out_c), _p(occ), _p(par), _p(slot), _p(cnt), _p(ws), ws.numel(), _s(),
          work={'bytes': 16.0 * n})  # lower bound: input coords only (outputs depend on the parent count)
    return out_c, occ, par, slot, cnt


def upsample(coords, occ, n_child=None, shift_add=None, want_coords=True):
    """Children of occupied bits.  n_child (host int) avoids the sync; else it is read back."""
    _need(coords, torch.int32, 'coords', 2)
    _need(occ, torch.uint8, 'occ', 1)
    n, dev = coords.shape[0], coords.device
    cap = 8 * n if n_child is None else n_child
    cc = torch.empty((cap, 4), dtype=torch.int32, device=dev) if want_coords else None
    par = torch.empty(cap, dtype=torch.int32, device=dev)
    slot = torch.empty(cap, dtype=torch.uint8, device=dev)
    cnt = torch.empty(1, dtype=torch.int32, device=dev)
    ws = workspace(_lib.load().fpcc_scan_workspace(n), dev)
    _call('fpcc_upsample', _p(coords), _p(occ), n, _p(cc), _p(par), _p(slot), _p(cnt), _p(shift_add), _p(ws), ws.numel(), _s())
    if n_child is None:
        n_child = int(cnt.item())
        cc = cc[:n_child] if cc is not None else None
        par, slot = par[:n_child], slot[:n_child]
    return cc, par, slot, n_child


def occ_to_bits(occ):
    out = torch.empty((occ.shape[0], 8), dtype=torch.int32, device=occ.device)
    _call('fpcc_occ_to_bits', _p(occ), occ.shape[0], _p(out), _s())
    return out


def slot_table(child_parent, child_slot):
    """k-major child-slot table [8, n_child]: parent row + 1 in the row of the child's slot, 0 elsewhere."""
    n = child_parent.shape[0]
    table = torch.empty((8, n), dtype=torch.int32, device=child_parent.device)
    _call('fpcc_slot_table', _p(child_parent), _p(child_slot), n, _p(table), n, _s())
    return table


def slot_pairs(child_parent, child_slot):
    """Pair lists grouped by child slot for the selection linear: (sel_row, sel_out, offsets[9])."""
    return kmap_compact(slot_table(child_parent, child_slot))


def kmap_transpose(table, n_in):
    """Transposed k-major neighbour table [kvol, n_in]: tt[k, j] = m + 1 where table[k, m] == j + 1, 0 elsewhere (the
    map of the dgrad).  Every (offset, input row) pair must have at most one output row (fpcc_kmap_transpose)."""
    _need(table, torch.int32, 'table', 2)
    kv, n_out = table.shape
    tt = torch.empty((kv, n_in), dtype=torch.int32, device=table.device)
    _call('fpcc_kmap_transpose', _p(table), kv, n_out, n_out, int(n_in), _p(tt), int(n_in), _s(),
          work={'bytes': 4.0 * kv * n_out + 4.0 * kv * n_in + 4.0 * int(torch.count_nonzero(table).item()) if _prof is not None else 0.0})
    return tt


def gather_patches(feats, table, kp):
    """im2col of a thin (C_in = 1 / 8) input along the neighbour table -> int8 [n_out, kp]"""
    _need(feats, torch.int8, 'feats', 2)
    _need(table, torch.int32, 'table', 2)
    kv, n_out = table.shape
    c = feats.shape[1]
    alloc = torch.empty if kp == kv * c else torch.zeros
    out = alloc((n_out, kp), dtype=torch.int8, device=feats.device)
    _call('fpcc_gather_patches', _p(feats), c, _p(table), n_out, kv, n_out, _p(out), kp, _s(),
          work={'bytes': float(n_out) * kv * (4 + c)})  # table read + patch bytes written
    return out


def morton_encode(xyz_rows, col0=1, msb_axis=0):
    """Morton codes of columns col0..col0+2 of an int32 [n, ld] tensor."""
    _need(xyz_rows, torch.int32, 'xyz', 2)
    n, ld = xyz_rows.shape
    codes = torch.empty(n, dtype=torch.int64, device=xyz_rows.device)
    _call('fpcc_morton_encode', xyz_rows.data_ptr() + 4 * col0, ld, n, msb_axis, _p(codes), _s())
    return codes


def occ_bits_q8(occ, q0, q1, out):
    """the 8 occupancy-bit channels (already requantised to the int8 levels q0 / q1) + 8 zero bytes into the 16-column slice
    `out` of a [rows, C + 16] int8 buffer (fpcc_occ_bits_q8)"""
    _need(occ, torch.uint8, 'occ', 1)
    if out.dtype != torch.int8 or out.dim() != 2 or out.shape != (occ.shape[0], 16) or out.stride(1) != 1:
        raise RuntimeError('occ_bits_q8: out must be an int8 [rows, 16] column slice')
    _call('fpcc_occ_bits_q8', _p(occ), occ.shape[0], int(q0), int(q1), out.data_ptr(), out.stride(0), _s(), work={'bytes': 17.0 * occ.shape[0]})
    return out


def gather_rows(rows, idx):
    """rows[idx] for an int32 [n, 4] coordinate tensor and an int64 permutation (the result of torch.argsort)."""
    _need(rows, torch.int32, 'rows', 2)
    _need(idx, torch.int64, 'index', 1)
    if rows.shape[1] != 4:
        raise RuntimeError('gather_rows: rows of 4 int32 expected')
    out = torch.empty((idx.shape[0], 4), dtype=torch.int32, device=rows.device)
    _call('fpcc_gather_rows16', _p(rows), _p(idx), idx.shape[0], _p(out), _s(), work={'bytes': 40.0 * idx.shape[0]})
    return out


# ---------------------------------------------------------------------------------------------
# GEMMs and epilogues
# ---------------------------------------------------------------------------------------------

def requant(inp, ep, out=None):
    _need(inp, torch.int32, 'input', 2)
    if inp.shape[0] <= 0 or inp.shape[1] <= 0:
        raise RuntimeError('requant: N > 0 && Ch > 0')
    work = ({'bytes': float(inp.numel() * 4 + inp.numel() * _OUT_DTYPE[ep.out_type].itemsize), 'desc': f'{inp.shape[0]}x{inp.shape[1]} out{ep.out_type}'}
            if _prof is not None else None)
    if out is not None and not out.is_contiguous():
        # a column slice of a wider int8 buffer (the two halves of a concatenation): rows at the buffer's pitch
        if out.dtype != torch.int8 or out.dim() != 2 or tuple(out.shape) != tuple(inp.shape) or out.stride(1) != 1:
            raise RuntimeError('requant: a strided output must be an int8 [rows, ch] column slice')
        _call('fpcc_requant_ld', _p(inp), inp.shape[0], inp.shape[1], C.byref(ep), out.data_ptr(), out.stride(0), _s(), tag='fpcc_requant', work=work)
        return out
    out = torch.empty(inp.shape, dtype=_OUT_DTYPE[ep.out_type], device=inp.device) if out is None else out
    _call('fpcc_requant', _p(inp), inp.shape[0], inp.shape[1], C.byref(ep), _p(out), _s(), work=work)
    return out


def prelu_i32(inp, slope):
    _need(inp, torch.int32, 'input', 2)
    _need(slope, torch.int32, 'slope')
    out = torch.empty_like(inp)
    _call('fpcc_prelu_i32', _p(inp), inp.numel(), _p(slope), _p(out), _s())
    return out


_POPC8 = {}


def kmap_from_parent(coarse_table, coarse_occ, parent, slot):
    """3x3x3 same-stride neighbour table of a level from its parent level's table (see fpcc_kmap_from_parent)."""
    _need(coarse_table, torch.int32, 'coarse table', 2)
    _need(coarse_occ, torch.uint8, 'coarse occupancy', 1)
    _need(parent, torch.int32, 'parent', 1)
    _need(slot, torch.uint8, 'slot', 1)
    if coarse_table.shape[0] != 27 or coarse_table.shape[1] != coarse_occ.shape[0] or parent.shape[0] != slot.shape[0]:
        raise RuntimeError('kmap_from_parent: shape mismatch')
    dev = coarse_table.device
    lut = _POPC8.get(dev.index)
    if lut is None:
        with cache_lock:
            lut = _POPC8.get(dev.index)
            if lut is None:
                lut = torch.tensor([bin(v).count('1') for v in range(256)], dtype=torch.int32, device=dev)
                publish_ready(dev)  # shared by every stream from here on (concurrent coding groups)
                _POPC8[dev.index] = lut
    cnt = lut[coarse_occ.long()]
    base = (torch.cumsum(cnt, 0, dtype=torch.int32) - cnt).contiguous()
    n_c, n_f = coarse_occ.shape[0], parent.shape[0]
    table = torch.empty((27, n_f), dtype=torch.int32, device=dev)
    _call('fpcc_kmap_from_parent', _p(coarse_table), n_c, n_c, _p(coarse_occ), _p(base), _p(parent), _p(slot), n_f, _p(table), n_f, _s(),
          work={'bytes': 4.0 * 27 * n_f + 5.0 * n_f + 4.0 * 27 * n_c})  # table written + parent/slot + parent table read once
    return table


def _tile_offsets_of(table):
    """profiling only: sum over 128-row tiles of the number of offsets with a neighbour in the tile (= MMA steps run)"""
    kv, n = table.shape
    any_k = (table != 0)
    pad = (-n) % 128
    if pad:
        any_k = torch.nn.functional.pad(any_k, (0, pad))
    return float(any_k.view(kv, -1, 128).any(dim=2).sum().item())


def group_rows(table):
    """Regroups the columns (output rows) of a k-major neighbour table by neighbour pattern.

    -> (table_p, perm): table_p[:, j] = table[:, perm[j]], perm int32 [n_out] sorted by the pattern bit mask.
    `spconv(..., table_p, ..., row_perm=perm)` gives the results of `spconv(..., table, ...)` while the kernel,
    which can only skip an offset for a whole 128-row tile, meets tiles whose rows share their offsets."""
    _need(table, torch.int32, 'table', 2)
    kv, n_out = table.shape
    masks = torch.empty(n_out, dtype=torch.int32, device=table.device)
    _call('fpcc_kmap_row_masks', _p(table), kv, n_out, n_out, _p(masks), _s(), work={'bytes': 4.0 * kv * n_out + 4.0 * n_out})
    perm = torch.sort(masks, stable=True)[1].to(torch.int32)  # stable: neighbouring rows stay neighbours within a pattern
    table_p = torch.empty_like(table)
    _call('fpcc_kmap_permute', _p(table), kv, n_out, n_out, _p(perm), _p(table_p), n_out, _s(), work={'bytes': 8.0 * kv * n_out + 4.0 * n_out})
    return table_p, perm


def spconv(in_feats, weight, table, ep, zp_comp=None, out=None, row_perm=None):
    """Fused output-stationary sparse conv from a k-major neighbour table [kvol, n_out] (optionally regrouped
    by `group_rows`: pass its permutation as row_perm)."""
    _need(in_feats, torch.int8, 'in_feats', 2)
    _need(weight, torch.int8, 'weight', 3)
    _need(table, torch.int32, 'table', 2)
    kv, c_out, c_in = weight.shape
    if table.shape[0] != kv or in_feats.shape[1] != c_in:
        raise RuntimeError(f'spconv: shape mismatch weight {tuple(weight.shape)} table {tuple(table.shape)} feats {tuple(in_feats.shape)}')
    n_out = table.shape[1]
    out = torch.empty((n_out, c_out), dtype=_ep_out_dtype(ep), device=in_feats.device) if out is None else out
    tag = work = None
    if _prof is not None:
        tag = 'spconv_' + gemm_engine(c_in, c_out, kv, zp_comp is not None)
        pairs = _pairs_of(table)
        work = {'ops': 2.0 * pairs * c_in * c_out, 'mma_ops': 2.0 * ((n_out + 127) // 128 * 128) * kv * c_in * c_out,
                'exec_ops': 2.0 * 128 * _tile_offsets_of(table) * c_in * c_out,
                'bytes': float(in_feats.numel() + weight.numel() + out.numel() * out.element_size() + 4 * table.numel())}
    if row_perm is not None:
        _need(row_perm, torch.int32, 'row_perm', 1)
        if row_perm.numel() != n_out:
            raise RuntimeError('spconv: row_perm must have one entry per output row')
    _call('fpcc_spconv_i8', _p(in_feats), in_feats.shape[0], c_in, _p(weight), kv, c_out, _p(table), n_out, n_out,
          _p(row_perm), _p(zp_comp), C.byref(ep), _p(out), _s(), tag=tag, work=work)
    return out


def linear(a, weight, ep, sel=None, n_out_rows=None, out=None):
    """Fused int8 linear.  sel = (sel_row, sel_out, offsets) computes only the selected (row, block) pairs;
    weight is then [n_groups*n, k] and the result has n_out_rows rows of n columns."""
    _need(a, torch.int8, 'input', 2)
    _need(weight, torch.int8, 'weight', 2)
    m, k = a.shape
    if weight.shape[1] != k:
        raise RuntimeError(f'linear: K mismatch {tuple(a.shape)} x {tuple(weight.shape)}')
    if out is not None and not out.is_contiguous():
        # int8 rows into a column slice of a wider buffer (fpcc_epilogue::out_ld)
        if out.dtype != torch.int8 or _ep_out_dtype(ep) != torch.int8 or out.dim() != 2 or out.stride(1) != 1 or out.stride(0) % 16:
            raise RuntimeError('linear: a strided output must be an int8 column slice with a pitch that is a multiple of 16')
        ep.out_ld = out.stride(0)
    if sel is None:
        n = weight.shape[0]
        out = torch.empty((m, n), dtype=_ep_out_dtype(ep), device=a.device) if out is None else out
        _call('fpcc_linear_i8', _p(a), m, k, _p(weight), n, None, None, None, 1, 0, C.byref(ep), _p(out), _s(),
              tag='linear_' + gemm_engine(k, n) if _prof is not None else None,
              work={'ops': 2.0 * m * k * n, 'desc': f'{m}x{k}->{n} out{ep.out_type} rb{int(bool(ep.row_bias))}'})
    else:
        sel_row, sel_out, offsets = sel
        groups = offsets.numel() - 1
        n = weight.shape[0] // groups
        out = torch.empty((n_out_rows, n), dtype=_ep_out_dtype(ep), device=a.device) if out is None else out
        _call('fpcc_linear_i8', _p(a), m, k, _p(weight), n, _p(sel_row), _p(sel_out), _p(offsets), groups, n_out_rows,
              C.byref(ep), _p(out), _s(), tag='linear_sel_' + gemm_engine(k, n) if _prof is not None else None,
              work={'ops': 2.0 * n_out_rows * k * n, 'desc': f'{m}x{k}->{groups}x{n} rows{n_out_rows} out{ep.out_type}'})
    return out


def gemm_i8(a, b, c, d):
    _need(a, torch.int8, 'A', 2); _need(b, torch.int8, 'B', 2); _need(d, torch.int32, 'D', 2)
    m, k = a.shape
    n = b.shape[0]
    if b.shape[1] != k or d.shape[0] != m or d.shape[1] != n:
        raise RuntimeError('gemm_i8: shape mismatch')
    if c is None or c.numel() == 0:
        mode = 0
    elif c.dim() == 1 and c.numel() == n:
        mode = 1
    elif c.dim() == 2 and tuple(c.shape) == (m, n):
        mode = 2
    else:
        raise RuntimeError('gemm_i8: C must be (N,), (M,N) or empty')
    if mode:
        _need(c, torch.int32, 'C')
    _call('fpcc_gemm_i8', _p(a), _p(b), _p(c) if mode else None, mode, _p(d), m, n, k, _s())


def gather_gemm_scatter_i8(a, b, d, gather_idx, scatter_idx):
    _need(a, torch.int8, 'A', 2); _need(b, torch.int8, 'B', 2); _need(d, torch.int32, 'D', 2)
    _need(gather_idx, torch.int32, 'gather_idx', 1); _need(scatter_idx, torch.int32, 'scatter_idx', 1)
    L = gather_idx.numel()
    if scatter_idx.numel() != L or L > d.shape[0] or b.shape[1] != a.shape[1] or d.shape[1] != b.shape[0]:
        raise RuntimeError('gather_gemm_scatter_i8: shape mismatch')
    if L:
        _call('fpcc_gather_gemm_scatter_i8', _p(a), _p(b), _p(d), _p(gather_idx), _p(scatter_idx), L, b.shape[0], a.shape[1], _s())


# ---------------------------------------------------------------------------------------------
# entropy head + coders
# ---------------------------------------------------------------------------------------------

def as_u16(t):
    """integer tensor -> uint16 bit patterns (truncating), avoiding torch's sparse uint16 op coverage"""
    return t.to(torch.int16).view(torch.uint16)


def softmax_i32(x):
    _need(x, torch.int32, 'input', 2)
    if not (x.shape[0] > 0 and x.shape[1] > 1):
        raise RuntimeError('softmax_int32: N > 0 && C > 1')
    out = torch.empty(x.shape, dtype=torch.uint32, device=x.device)
    _call('fpcc_softmax_i32', _p(x), x.shape[0], x.shape[1], _p(out), _s())
    return out


def _logits_pitch(logits):
    """logits may be a column slice of a padded linear output: [n, s] with unit column stride and any row pitch"""
    if logits.dtype != torch.int32 or not logits.is_cuda or logits.dim() != 2:
        raise RuntimeError('logits: expected a 2-D int32 CUDA tensor')
    if logits.shape[0] > 1 and (logits.stride(1) != 1 or logits.stride(0) < logits.shape[1]):
        logits = logits.contiguous()
    return logits, (logits.stride(0) if logits.shape[0] > 1 else logits.shape[1])


def quantize_cdf(logits, ld=CDF_LD):
    logits, pitch = _logits_pitch(logits)
    n, s = logits.shape
    ld = max(ld, s)
    out = torch.empty((n, ld), dtype=torch.uint16, device=logits.device)
    _call('fpcc_quantize_cdf', _p(logits), pitch, n, s, _p(out), ld, _s(), work={'bytes': 4.0 * s * n + 2.0 * ld * n})
    return out


def cdf_symbol_ranges(logits, symbols, out=None):
    logits, pitch = _logits_pitch(logits)
    _need(symbols, torch.int32, 'symbols', 1)
    n, s = logits.shape
    out = torch.empty(n, dtype=torch.int32, device=logits.device) if out is None else out
    _call('fpcc_cdf_symbol_ranges', _p(logits), pitch, n, s, _p(symbols), _p(out), _s(), work={'bytes': 4.0 * s * n + 6.0 * n})
    return out


def table_symbol_ranges(cdf, symbols, out=None):
    _need(cdf, torch.uint16, 'cdf', 2)
    _need(symbols, torch.int32, 'symbols', 1)
    n = symbols.numel()
    out = torch.empty(n, dtype=torch.int32, device=cdf.device) if out is None else out
    if n:
        _call('fpcc_table_symbol_ranges', _p(cdf), cdf.shape[0], cdf.shape[1], _p(symbols), n, _p(out), _s())
    return out


def rans_encode(ranges, rng_off, out_stride, bits=None, out=None, state_io=None, flush=True, total=None):
    """-> (out uint8 [n_streams, out_stride], out_len int32 [n_streams]); stream b = out[b, out_stride-len:]"""
    _need(ranges, torch.int32, 'ranges', 1)  # packed uint32 bit patterns carried as int32
    _need(rng_off, torch.int64, 'rng_off', 1)
    ns = rng_off.numel() - 1
    if out is None:
        out = torch.empty((ns, out_stride), dtype=torch.uint8, device=ranges.device)
    out_len = torch.empty(ns, dtype=torch.int32, device=ranges.device)
    total = ranges.numel() if total is None else int(total)
    ws = workspace(16 * max(total, 1), ranges.device)
    _call('fpcc_rans_encode', _p(ranges), _p(bits), _p(rng_off), ns, total, _p(out), out_stride, _p(out_len),
          _p(state_io), 1 if flush else 0, _p(ws), ws.numel(), _s())
    return out, out_len


class RansDecodeStreams:
    """Device-resident decoder state for n streams (RansDecoder::flush + decode, batched)."""

    PAD = 512  # the decoder's byte window reads (and prefetches) ahead of the stream position

    def __init__(self, data, byte_off, byte_len, padded=False):
        _need(data, torch.uint8, 'bytes', 1)
        if not padded:
            data = torch.cat([data, torch.zeros(self.PAD, dtype=torch.uint8, device=data.device)])
        self.data, self.byte_off = data, byte_off
        self.n = byte_off.numel()
        self.state = torch.empty((self.n, 4), dtype=torch.int32, device=data.device)
        _call('fpcc_rans_dec_init', _p(self.state), _p(data), _p(byte_off), _p(byte_len), self.n, _s())

    def decode(self, cdf, s, row_off, n_rows, shared=False, rows_per_stream=False, s_per_stream=None):
        """cdf: uint16 [rows, ld] (one row per symbol), [1, s] shared by all streams, or [n_streams, ld] with
        rows_per_stream.  row_off int64 [n_streams+1] (device): symbol range of every stream."""
        _need(cdf, torch.uint16, 'cdf', 2)
        sym = torch.empty(n_rows, dtype=torch.int32, device=cdf.device)
        _call('fpcc_rans_decode', _p(self.state), _p(self.data), _p(self.byte_off), _p(cdf),
              1 if shared else cdf.shape[0], s, cdf.shape[1], _p(row_off), self.n, _p(sym),
              1 if rows_per_stream else 0, _p(s_per_stream), _s())
        return sym

    def error(self):
        return bool((self.state[:, 3] != 0).any().item())


# ---------------------------------------------------------------------------------------------
# fp16 / bf16 tensor-core path (float layer API)
# ---------------------------------------------------------------------------------------------
_F_DT = {torch.float16: 0, torch.bfloat16: 1}
_F_OUT = {torch.float16: 0, torch.bfloat16: 1, torch.float32: 2}
ACT_NONE, ACT_RELU, ACT_LEAKY = 0, 1, 2


def _fargs(bias, residual, out_dtype):
    if bias is not None:
        _need(bias, torch.float32, 'bias', 1)
    if residual is not None and residual.dtype != out_dtype:
        raise RuntimeError('residual must have the output dtype')
    return _p(bias), _p(residual)


def spconv_f16(feats, weight_t, table, bias=None, act=ACT_NONE, slope=0.0, residual=None, post_act=ACT_NONE,
               post_slope=0.0, out_dtype=None, row_perm=None):
    """Fused fp16/bf16 sparse conv: feats [n_in, c_in], weight_t [kvol, c_out, c_in] (same dtype), k-major table."""
    if feats.dtype not in _F_DT or weight_t.dtype != feats.dtype:
        raise RuntimeError(f'spconv_f16: fp16/bf16 features and weights of one dtype expected, got {feats.dtype}/{weight_t.dtype}')
    if not (feats.is_cuda and feats.is_contiguous() and weight_t.is_contiguous() and table.is_contiguous()):
        raise RuntimeError('spconv_f16: contiguous CUDA tensors expected')
    kv, c_out, c_in = weight_t.shape
    if table.shape[0] != kv or feats.shape[1] != c_in:
        raise RuntimeError('spconv_f16: shape mismatch')
    out_dtype = feats.dtype if out_dtype is None else out_dtype
    n_out = table.shape[1]
    out = torch.empty((n_out, c_out), dtype=out_dtype, device=feats.device)
    pb, pr = _fargs(bias, residual, out_dtype)
    work = None
    if _prof is not None:
        work = {'ops': 2.0 * _pairs_of(table) * c_in * c_out, 'mma_ops': 2.0 * ((n_out + 127) // 128 * 128) * kv * c_in * c_out}
    if row_perm is not None:
        _need(row_perm, torch.int32, 'row_perm', 1)
    _call('fpcc_spconv_f16', _p(feats), _F_DT[feats.dtype], feats.shape[0], c_in, _p(weight_t), kv, c_out, _p(table), n_out,
          n_out, _p(row_perm), pb, act, float(slope), pr, post_act, float(post_slope), _p(out), _F_OUT[out_dtype], _s(),
          tag='spconv_f16_tc', work=work)
    return out


WGRAD_CHUNK = 2048  # pairs per tile of fpcc_spconv_wgrad_f16 (csrc/igemm_tc.cu: WG_CHUNK)
_wgrad_tiles = {}


def wgrad_supported(c_in, c_out):
    """channel counts the tensor-core weight-gradient kernel takes (after padding to 128 / 256 x a multiple of 64)"""
    return c_in <= 256 and c_out <= 256


def spconv_wgrad_f16(x, dy, in_map, out_map, offsets_host, c_in, c_out):
    """dW[k] = x[in_k]^T @ dy[out_k] for every kernel offset on the tensor cores (fp32 accumulation, fp32 result
    [kvol, c_in, c_out]).  x [n_in, >= c_in], dy [n_out, >= c_out] fp16 / bf16; in_map / out_map / offsets_host: the
    compacted pair lists of `kmap_compact` (offsets as a host list)."""
    if x.dtype not in _F_DT or dy.dtype != x.dtype:
        raise RuntimeError('spconv_wgrad_f16: fp16/bf16 inputs of one dtype expected')
    if not wgrad_supported(c_in, c_out):
        raise RuntimeError('spconv_wgrad_f16: at most 256 input and output channels')
    kv = len(offsets_host) - 1
    c_in_p = 128 if c_in <= 128 else 256
    c_out_p = (c_out + 63) // 64 * 64
    xp = torch.nn.functional.pad(x[:, :c_in], (0, c_in_p - c_in)).contiguous() if x.shape[1] != c_in_p else x.contiguous()
    gp = torch.nn.functional.pad(dy[:, :c_out], (0, c_out_p - c_out)).contiguous() if dy.shape[1] != c_out_p else dy.contiguous()
    tkey = (tuple(int(o) for o in offsets_host), x.device.index)
    tl = _wgrad_tiles.get(tkey)
    if tl is None:  # the tile list of a kernel map is the same for every layer and step that uses the map
        tiles = []
        for k in range(kv):
            s, e = int(offsets_host[k]), int(offsets_host[k + 1])
            for b in range(s, e, WGRAD_CHUNK):
                tiles.append((k, b, min(e, b + WGRAD_CHUNK), 0))
        tl = torch.tensor(tiles, dtype=torch.int32).reshape(-1, 4).to(x.device)
        if len(_wgrad_tiles) >= 64:
            _wgrad_tiles.pop(next(iter(_wgrad_tiles)))
        _wgrad_tiles[tkey] = tl
    dw = torch.zeros((kv, c_in, c_out), dtype=torch.float32, device=x.device)
    if tl.shape[0]:
        n_pairs = int(offsets_host[-1])
        _call('fpcc_spconv_wgrad_f16', _p(xp), _p(gp), _F_DT[x.dtype], c_in_p, c_out_p, _p(in_map), _p(out_map), _p(tl), tl.shape[0],
              _p(dw), c_in, c_out, _s(), tag='spconv_wgrad_tc', work={'ops': 2.0 * n_pairs * c_in * c_out})
    return dw


def act_grad_f16(dy, y, act, slope, c_pad, out_dtype=None, want_bias=True):
    """Backward of an activation fused into the conv / linear epilogue (fpcc_act_grad_f16), one pass:
    -> (dz [n, c_pad] in out_dtype (default: y's dtype, fp16 / bf16) with zero pad columns, dbias fp32 [c] | None).
    dy, y: [n, c] fp16 / bf16 / fp32 with unit column stride (y = the forward output; unused for ACT_NONE)."""
    n, c = dy.shape
    out_dtype = (y.dtype if y is not None and y.dtype != torch.float32 else torch.float16) if out_dtype is None else out_dtype
    if out_dtype not in _F_DT:
        raise RuntimeError(f'act_grad_f16: dz must be fp16 or bf16, got {out_dtype}')
    for t, name in ((dy, 'dy'), (y, 'y')):
        if t is None:
            continue
        if t.dtype not in _F_OUT or not t.is_cuda or t.dim() != 2 or tuple(t.shape) != (n, c):
            raise RuntimeError(f'act_grad_f16: {name} must be a 2-D fp16 / bf16 / fp32 CUDA tensor of shape {(n, c)}')
    rows = lambda t: t if t.stride(1) == 1 and t.stride(0) >= c else t.contiguous()  # noqa: E731  (any row pitch >= c)
    dy = rows(dy)
    y = rows(y) if y is not None else None
    dz = torch.empty((n, c_pad), dtype=out_dtype, device=dy.device)
    db = torch.empty(c, dtype=torch.float32, device=dy.device) if want_bias else None
    ws = workspace(_lib.load().fpcc_act_grad_workspace(n, c), dy.device) if want_bias else None
    ld_y = y.stride(0) if y is not None else c
    nbytes = float(n) * c * (dy.element_size() + (y.element_size() if (y is not None and act != ACT_NONE) else 0)) + float(n) * c_pad * dz.element_size()
    _call('fpcc_act_grad_f16', _p(dy), _F_OUT[dy.dtype], dy.stride(0), _p(y), _F_OUT[y.dtype] if y is not None else 0,
          ld_y, n, c, int(act), float(slope), _p(dz), _F_DT[out_dtype], int(c_pad), _p(db), _p(ws), 0 if ws is None else ws.numel(), _s(),
          work={'bytes': nbytes})
    return dz, db


def linear_f16(a, weight, bias=None, act=ACT_NONE, slope=0.0, residual=None, post_act=ACT_NONE, post_slope=0.0,
               out_dtype=None, sel=None, n_out_rows=None, out=None):
    """Fused fp16/bf16 linear: a [m, k], weight [n_groups*n, k]; sel = (sel_row, sel_out, offsets) as in `linear`."""
    if a.dtype not in _F_DT or weight.dtype != a.dtype:
        raise RuntimeError('linear_f16: fp16/bf16 inputs of one dtype expected')
    if not (a.is_cuda and a.is_contiguous() and weight.is_contiguous()):
        raise RuntimeError('linear_f16: contiguous CUDA tensors expected')
    m, k = a.shape
    out_dtype = a.dtype if out_dtype is None else out_dtype
    if sel is None:
        n = weight.shape[0]
        out = torch.empty((m, n), dtype=out_dtype, device=a.device)
        pb, pr = _fargs(bias, residual, out_dtype)
        _call('fpcc_linear_f16', _p(a), _F_DT[a.dtype], m, k, _p(weight), n, None, None, None, 1, 0, pb, act, float(slope), pr,
              post_act, float(post_slope), _p(out), _F_OUT[out_dtype], _s(), tag='linear_f16_tc', work={'ops': 2.0 * m * k * n})
    else:
        sel_row, sel_out, offsets = sel
        groups = offsets.numel() - 1
        n = weight.shape[0] // groups
        out = torch.empty((n_out_rows, n), dtype=out_dtype, device=a.device) if out is None else out
        pb, pr = _fargs(bias, residual, out_dtype)
        _call('fpcc_linear_f16', _p(a), _F_DT[a.dtype], m, k, _p(weight), n, _p(sel_row), _p(sel_out), _p(offsets), groups,
              n_out_rows, pb, act, float(slope), pr, post_act, float(post_slope), _p(out), _F_OUT[out_dtype], _s(),
              tag='linear_sel_f16_tc', work={'ops': 2.0 * n_out_rows * k * n})
    return out


# ---------------------------------------------------------------------------------------------
# deep-factorized entropy model (csrc/entropy_model.cu)
# ---------------------------------------------------------------------------------------------
def _em_rows(t, c, name):
    if t.dtype != torch.float32 or not t.is_cuda or t.dim() != 2 or t.shape[1] != c:
        raise RuntimeError(f'factorized entropy model: {name} must be a 2-D fp32 CUDA tensor with {c} columns')
    return t if t.stride(1) == 1 and t.stride(0) >= c else t.contiguous()  # any row pitch >= c


def _em_params(params):
    if params.dtype != torch.float32 or not params.is_cuda or params.dim() != 2 or params.shape[1] != 43:
        raise RuntimeError('factorized entropy model: params must be an fp32 CUDA tensor [C, 43]')
    return params.contiguous()


def factorized_bits(y, params, bound=1e-9):
    """-log2(max(L_c(y), bound)) per element: y fp32 [n, C], params fp32 [C, 43] -> bits fp32 [n, C]"""
    params = _em_params(params)
    n, c = y.shape[0], params.shape[0]
    y = _em_rows(y, c, 'y')
    bits = torch.empty((n, c), dtype=torch.float32, device=y.device)
    _call('fpcc_factorized_bits', _p(y), y.stride(0), n, c, _p(params), float(bound), _p(bits), _s(),
          work={'bytes': 8.0 * n * c + 172.0 * c})
    return bits


def factorized_grad(y, params, dbits, bound=1e-9):
    """-> (dy fp32 [n, C], dparams fp32 [C, 43]) of sum(dbits * factorized_bits(y, params)); dparams with respect to the
    raw params, reproducible bit for bit"""
    params = _em_params(params)
    n, c = y.shape[0], params.shape[0]
    y, dbits = _em_rows(y, c, 'y'), _em_rows(dbits, c, 'dbits')
    if dbits.shape[0] != n:
        raise RuntimeError('factorized entropy model: dbits must have the rows of y')
    dy = torch.empty((n, c), dtype=torch.float32, device=y.device)
    dp = torch.empty((c, 43), dtype=torch.float32, device=y.device)
    ws = workspace(_lib.load().fpcc_factorized_grad_workspace(n, c), y.device)
    _call('fpcc_factorized_grad', _p(y), y.stride(0), _p(dbits), dbits.stride(0), n, c, _p(params), float(bound), _p(dy), _p(dp),
          _p(ws), ws.numel(), _s(), work={'bytes': 12.0 * n * c + 344.0 * c})
    return dy, dp


def factorized_pmf(params, lo=-64, n_sym=129):
    """pmf fp64 [C, n_sym]: pmf[c, k] = L_c(lo + k), by the device function of factorized_bits"""
    params = _em_params(params)
    pmf = torch.empty((params.shape[0], n_sym), dtype=torch.float64, device=params.device)
    _call('fpcc_factorized_pmf', _p(params), params.shape[0], int(lo), int(n_sym), _p(pmf), _s())
    return pmf
