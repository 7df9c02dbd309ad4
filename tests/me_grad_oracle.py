"""Dense fp64 restatement of the MinkowskiEngine-shim layers for gradient checks (CPU, torch autograd): the forward of
each layer kind written with plain indexing on the neighbour tables of `oracle.float_ops.me_lookup`, so that
`torch.autograd.grad` through it gives reference d_feats / d_kernel / d_bias for the tcgen05 backward of
`fastpcc_b200/autograd.py`.  Also the torch reference of the transposed neighbour table (`fpcc_kmap_transpose`) and of
the fused-activation backward (`fpcc_act_grad_f16`)."""
import numpy as np
import torch

from oracle import float_ops as FO

ACT_NONE, ACT_RELU, ACT_LEAKY = 0, 1, 2


def transpose_table(table: torch.Tensor, n_in: int) -> torch.Tensor:
    """tt[k, j] = m + 1 where table[k, m] == j + 1, 0 elsewhere (nonzero + scatter)"""
    kv, n_out = table.shape
    tt = torch.zeros((kv, n_in), dtype=torch.int32, device=table.device)
    k_idx, m_idx = torch.nonzero(table, as_tuple=True)
    tt[k_idx, (table[k_idx, m_idx] - 1).long()] = (m_idx + 1).to(torch.int32)
    return tt


def act(x, code, slope, mask=None):
    """mask (bool, optional): where the activation passes x unchanged.  A test passes the sign pattern of the forward
    output under test, so that a pre-activation within rounding of the kink takes the same branch in both."""
    if mask is not None and code != ACT_NONE:
        return torch.where(mask, x, x * (slope if code == ACT_LEAKY else 0.0))
    if code == ACT_RELU:
        return torch.relu(x)
    if code == ACT_LEAKY:
        return torch.where(x > 0, x, x * slope)
    return x


def act_grad(dy, y, code, slope, c_pad, dtype):
    """-> (dz [n, c_pad] rounded once from fp32 to dtype, zero pad columns; dbias fp64 [c])"""
    g = dy.float()
    if code != ACT_NONE:
        g = g * torch.where(y.float() > 0, torch.ones_like(g), torch.full_like(g, slope))
    dz = torch.zeros((g.shape[0], c_pad), dtype=dtype, device=g.device)
    dz[:, :g.shape[1]] = g.to(dtype)
    return dz, g.double().sum(0)


def table(in_coords: torch.Tensor, out_coords: torch.Tensor, kernel_size, scale) -> torch.Tensor:
    """k-major [K, n_out] (input row + 1 | 0) in ME's offset convention"""
    s = np.broadcast_to(np.asarray(scale, dtype=np.int64), (3,))
    return torch.from_numpy(FO.me_lookup(in_coords.cpu().numpy(), out_coords.cpu().numpy(), tuple(kernel_size), s)).long()


def conv(f, w, b, t, code=ACT_NONE, slope=0.0, mask=None):
    """out[o] = act(sum_k f[t[k, o] - 1] @ w[k] + b); f [n_in, C_in], w [K, C_in, C_out], t k-major [K, n_out]"""
    out = torch.zeros((t.shape[1], w.shape[2]), dtype=f.dtype)
    for k in range(t.shape[0]):
        o = torch.nonzero(t[k]).reshape(-1)
        if o.numel():
            out = out.index_add(0, o, f[t[k, o] - 1] @ w[k])
    if b is not None:
        out = out + b.reshape(1, -1)
    return act(out, code, slope, mask)


def tconv(f, w, b, in_coords, out_coords, tensor_stride, code=ACT_NONE, slope=0.0, mask=None):
    """k2s2 transposed conv onto existing finer coordinates: out[child] = act(f[parent] @ w[slot] + b), act(b) for orphans"""
    oc = out_coords.cpu().long()
    par_c = oc.clone()
    par_c[:, 1:] = torch.div(oc[:, 1:], tensor_stride, rounding_mode='floor') * tensor_stride
    par = table(in_coords, par_c, (1, 1, 1), 1)[0]
    d = (oc[:, 1:] - par_c[:, 1:]) // (tensor_stride // 2)
    slot = d[:, 0] + 2 * d[:, 1] + 4 * d[:, 2]
    t = torch.zeros((8, oc.shape[0]), dtype=torch.long)
    rows = torch.nonzero(par).reshape(-1)
    t[slot[rows], rows] = par[rows]
    return conv(f, w, b, t, code, slope, mask)


def gen(f, w, b, code=ACT_NONE, slope=0.0, mask=None):
    """generative k2s2: out[8n + k] = act(f[n] @ w[k] + b)"""
    out = torch.einsum('ni,kio->nko', f, w).reshape(-1, w.shape[2])
    if b is not None:
        out = out + b.reshape(1, -1)
    return act(out, code, slope, mask)
