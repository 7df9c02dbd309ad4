"""torch-CPU fp32 restatement of the float operators behind the MinkowskiEngine-shaped layer API, under the SAME
function names as fastpcc_b200/ops.py (the slice fastpcc_b200/me.py calls) -- TEST INFRASTRUCTURE ONLY.

oracle/me_cpu.py binds these in place of the CUDA front-end, which turns the shim's coordinate bookkeeping into a CPU
MinkowskiEngine stand-in on which the reference's UNMODIFIED float codecs (lossy_coord_v2 ...) run in this container:
that run is the float oracle of the "+ lossy codec" row (bpp / D1-PSNR fixtures in tests/golden).  Semantics are
those of oracle/float_ops.py (ME's published conventions as pinned by the reference's call sites): parity unpinned
against ME itself, which cannot be installed offline.
"""
import numpy as np
import torch

from fastpcc_b200.ops import f16_weight, f16_widths, pad_cols  # noqa: F401  operand padding: bookkeeping, not arithmetic
from . import float_ops as F

ACT_NONE, ACT_RELU, ACT_LEAKY = 0, 1, 2


def _split3(a):
    x = a.astype(np.uint64) & np.uint64(0x1fffff)
    x = (x | (x << np.uint64(32))) & np.uint64(0x1f00000000ffff)
    x = (x | (x << np.uint64(16))) & np.uint64(0x1f0000ff0000ff)
    x = (x | (x << np.uint64(8))) & np.uint64(0x100f00f00f00f00f)
    x = (x | (x << np.uint64(4))) & np.uint64(0x10c30c30c30c30c3)
    x = (x | (x << np.uint64(2))) & np.uint64(0x1249249249249249)
    return x


def morton_encode(xyz_rows, col0=1, msb_axis=0):
    """morton3d.cu:19-37: msb_axis 0 -> x most significant, 2 -> z most significant"""
    c = xyz_rows.numpy()[:, col0:col0 + 3]
    a, b, d = (c[:, 2], c[:, 1], c[:, 0]) if msb_axis == 0 else (c[:, 0], c[:, 1], c[:, 2])
    code = _split3(a) | (_split3(b) << np.uint64(1)) | (_split3(d) << np.uint64(2))
    return torch.from_numpy(code.astype(np.int64))


def hash_build(coords, layout=0, keys=None, vals=None):
    return coords, None  # the "table" is the coordinate list itself


def kmap_lookup(keys, vals, out_coords, kernel_size, stride, layout=0, k_major=True, pad_rows=None, convention=0):
    assert convention == 1 and k_major, 'the CPU stand-in only serves the ME convention'
    scale = np.asarray(stride, dtype=np.int64)
    return torch.from_numpy(F.me_lookup(keys.numpy(), out_coords.numpy(), tuple(kernel_size), scale))


def kmap_compact(table, omit_k=-1):
    t = table.numpy()
    ins, outs, off = [], [], [0]
    for k in range(t.shape[0]):
        o = np.nonzero(t[k])[0] if k != omit_k else np.zeros(0, np.int64)
        ins.append(t[k, o] - 1)
        outs.append(o)
        off.append(off[-1] + o.size)
    cat = lambda xs: torch.from_numpy(np.concatenate(xs).astype(np.int32)) if xs else torch.zeros(0, dtype=torch.int32)  # noqa: E731
    return cat(ins), cat(outs), torch.tensor(off, dtype=torch.int32)


def group_rows(table):
    return table, torch.arange(table.shape[1], dtype=torch.int32)  # no tiles on the CPU: identity grouping


def slot_pairs(child_parent, child_slot):
    """pairs (parent row, child row) grouped by child slot 0..7 -> (sel_row, sel_out, offsets[9]); slot 255 joins no group"""
    par, slot = child_parent.numpy(), child_slot.numpy()
    rows, outs, off = [], [], [0]
    for g in range(8):
        o = np.nonzero(slot == g)[0]
        rows.append(par[o])
        outs.append(o)
        off.append(off[-1] + o.size)
    return (torch.from_numpy(np.concatenate(rows).astype(np.int32)), torch.from_numpy(np.concatenate(outs).astype(np.int32)),
            torch.tensor(off, dtype=torch.int32))


def _act(x, code, slope):
    if code == ACT_RELU:
        return torch.relu(x)
    if code == ACT_LEAKY:
        return torch.where(x < 0, x * slope, x)
    return x


def linear_f16(a, weight, bias=None, act=ACT_NONE, slope=0.0, residual=None, post_act=ACT_NONE, post_slope=0.0,
               out_dtype=None, sel=None, n_out_rows=None, out=None):
    a, w = a.float(), weight.float()
    if sel is None:
        y = a @ w.T
        if bias is not None:
            y = y + bias[None]
        y = _act(y, act, slope)
        if residual is not None:
            y = _act(y + residual.float(), post_act, post_slope)
        return y
    sel_row, sel_out, offsets = sel
    off = offsets.tolist()
    n = w.shape[0] // (len(off) - 1)
    res = out.float().clone() if out is not None else torch.zeros((n_out_rows, n))
    for g in range(len(off) - 1):
        if off[g + 1] > off[g]:
            r, o = sel_row[off[g]: off[g + 1]].long(), sel_out[off[g]: off[g + 1]].long()
            y = a[r] @ w[g * n: (g + 1) * n].T
            if bias is not None:
                y = y + bias[None]
            res[o] = _act(y, act, slope)
    return res


def spconv_f16(feats, weight_t, table, bias=None, act=ACT_NONE, slope=0.0, residual=None, post_act=ACT_NONE,
               post_slope=0.0, out_dtype=None, row_perm=None):
    """weight_t [K, C_out, C_in]; table k-major [K, n_out] (input row + 1 | 0); offsets accumulate in ascending k"""
    f, w = feats.float(), weight_t.float()
    t = table.long()
    y = torch.zeros((t.shape[1], w.shape[1]))
    for k in range(t.shape[0]):
        o = torch.nonzero(t[k]).reshape(-1)
        if o.numel():
            y[o] += f[t[k, o] - 1] @ w[k].T
    if bias is not None:
        y = y + bias[None]
    y = _act(y, act, slope)
    if residual is not None:
        y = _act(y + residual.float(), post_act, post_slope)
    if row_perm is not None:
        out = torch.empty_like(y)
        out[row_perm.long()] = y
        y = out
    return y
