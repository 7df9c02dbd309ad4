"""Float64 torch restatement of the fp16 / bf16 tensor-core GEMMs of csrc/igemm_tc.cu (fpcc_spconv_f16,
fpcc_linear_f16 dense and selection form, fpcc_spconv_wgrad_f16), the textbook error bound of their fp32 accumulation,
the neighbour-table builders the device tests drive them with, and a pairwise covering design for the test matrix.

Everything here is plain tensor code that runs on any device: the device tests evaluate it on the GPU in fp64, the
host tests on the CPU.  Tables are k-major [kvol, >= n_out] with entry = input row + 1 and 0 = no neighbour, as in the
header; column j of a table describes output row j."""
import itertools
import random

import torch

ACT_NONE, ACT_RELU, ACT_LEAKY = 0, 1, 2
TC_M = 128          # output rows per tile of the persistent kernel
EXACT_LIMIT = 2 ** 20  # sums of |terms| below this add exactly in fp32 in any order (with slopes >= 1/4 twice: 24 bits)


def act(x, code, slope):
    if code == ACT_RELU:
        return torch.relu(x)
    if code == ACT_LEAKY:
        return torch.where(x < 0, x * slope, x)
    return x


def epilogue(acc, bias=None, code=ACT_NONE, slope=0.0, residual=None, post_act=ACT_NONE, post_slope=0.0):
    """v = acc + bias; v = act(v); [v += residual]; v = post_act(v) in fp64 (post_act applies with or without a residual)"""
    v = acc if bias is None else acc + bias.double().reshape(1, -1)
    v = act(v, code, slope)
    if residual is not None:
        v = v + residual.double()
    return act(v, post_act, post_slope)


def conv_acc(feats, w_t, table, absolute=False):
    """acc[o] = sum_k feats[table[k, o] - 1] @ w_t[k]^T over the entries != 0; w_t [kvol, C_out, C_in].  Only the
    gathered rows are widened to fp64, so `feats` may be larger than the device could hold in fp64.  absolute: the same
    sum over |feats| and |w_t|."""
    w = w_t.double().abs() if absolute else w_t.double()
    kv, n_out = table.shape
    acc = torch.zeros((n_out, w.shape[1]), dtype=torch.float64, device=feats.device)
    for k in range(kv):
        o = torch.nonzero(table[k]).reshape(-1)
        if o.numel():
            rows = feats[table[k, o].long() - 1].double()
            acc.index_add_(0, o, (rows.abs() if absolute else rows) @ w[k].t())
    return acc


def spconv(feats, w_t, table, bias=None, code=ACT_NONE, slope=0.0, residual=None, post_act=ACT_NONE, post_slope=0.0):
    """fpcc_spconv_f16: out [n_out, C_out] fp64"""
    return epilogue(conv_acc(feats, w_t, table), bias, code, slope, residual, post_act, post_slope)


def linear(a, w, bias=None, code=ACT_NONE, slope=0.0, residual=None, post_act=ACT_NONE, post_slope=0.0):
    """dense fpcc_linear_f16: out = epilogue(a @ w^T), w [n, k]"""
    return epilogue(a.double() @ w.double().t(), bias, code, slope, residual, post_act, post_slope)


def linear_sel(a, w, sel_row, sel_out, offsets, out, bias=None, code=ACT_NONE, slope=0.0, residual=None,
               post_act=ACT_NONE, post_slope=0.0):
    """selection fpcc_linear_f16: for the pairs i of group g (offsets[g] <= i < offsets[g+1])
        out[sel_out[i]] = epilogue(a[sel_row[i]] @ w[g n : g n + n]^T)
    with the bias per column, shared by the groups, and the residual row of the OUTPUT row.  Rows of `out` that no pair
    selects keep their values.  -> fp64 copy of `out` with the selected rows written."""
    n = out.shape[1]
    res = out.double().clone()
    off = [int(v) for v in offsets]
    for g in range(len(off) - 1):
        s, e = off[g], off[g + 1]
        if e <= s:
            continue
        ro, ri = sel_out[s:e].long(), sel_row[s:e].long()
        acc = a.double()[ri] @ w.double()[g * n:(g + 1) * n].t()
        r = residual[ro] if residual is not None else None
        res[ro] = epilogue(acc, bias, code, slope, r, post_act, post_slope)
    return res


def wgrad(x, dy, in_map, out_map, offsets):
    """fpcc_spconv_wgrad_f16: dW[k] = x[in_k]^T @ dy[out_k] over the pairs offsets[k] .. offsets[k+1]; fp64 [kvol, C_in, C_out]"""
    off = [int(v) for v in offsets]
    dw = torch.zeros((len(off) - 1, x.shape[1], dy.shape[1]), dtype=torch.float64, device=x.device)
    for k in range(len(off) - 1):
        s, e = off[k], off[k + 1]
        if e > s:
            dw[k] = x.double()[in_map[s:e].long()].t() @ dy.double()[out_map[s:e].long()]
    return dw


def abs_sum(feats, w_t, table, bias=None, residual=None):
    """S = sum |a w| over the product terms of every output element, + |b| (+ |res|): fp64 [n_out, C_out]"""
    s = conv_acc(feats, w_t, table, absolute=True)
    if bias is not None:
        s = s + bias.double().abs().reshape(1, -1)
    if residual is not None:
        s = s + residual.double().abs()
    return s


def bound(s, n_terms):
    """Worst-case |got - ref| of an fp32 result whose n_terms product terms (plus bias, activation and residual steps)
    are summed in any order, with round-to-nearest or truncation: 2 n u S with u = 2^-24 and n = n_terms + 3."""
    return 2.0 * (n_terms + 3) * 2.0 ** -24 * s


def assert_exact_premise(s):
    """The integer-exact tests rely on every partial sum being an integer (or a dyadic rational of few bits) below 2^24;
    this asserts the sufficient condition sum |terms| < 2^20 instead of assuming it."""
    m = float(s.max()) if s.numel() else 0.0
    assert m < EXACT_LIMIT, f'integer-exact premise violated: sum |terms| = {m} >= 2^20'


# ---- neighbour tables ------------------------------------------------------------------------------------------------
def _gen(seed):
    g = torch.Generator()
    g.manual_seed(seed)
    return g


def random_table(kvol, n_out, n_in, p, seed):
    """each entry present with probability p, sources uniform over the n_in input rows"""
    g = _gen(seed)
    src = torch.randint(1, n_in + 1, (kvol, n_out), generator=g, dtype=torch.int32)
    return torch.where(torch.rand((kvol, n_out), generator=g) < p, src, torch.zeros_like(src))


def empty_tile_table(kvol, n_out, n_in, p, seed):
    """random table in which whole 128-row tiles have no neighbour at all: tile 1 and every 7th tile after it, between
    active tiles (one tile: the whole table is empty; two tiles: the second one)"""
    t = random_table(kvol, n_out, n_in, p, seed)
    n_tiles = (n_out + TC_M - 1) // TC_M
    for i in range(min(1, n_tiles - 1), n_tiles, 7):
        t[:, i * TC_M:(i + 1) * TC_M] = 0
    return t


def one_row_per_offset_table(kvol, n_out, n_in, seed):
    """in every tile each offset is active in exactly one row, and those rows are spread over all four 32-row
    producer warps of the tile: the offset mask of a tile exists only as the OR over the warps"""
    g = _gen(seed)
    t = torch.zeros((kvol, n_out), dtype=torch.int32)
    for tile in range(0, n_out, TC_M):
        rows = min(TC_M, n_out - tile)
        for k in range(kvol):
            r = ((k % 4) * 32 + (5 * k + tile // TC_M) % 32) % rows
            t[k, tile + r] = int(torch.randint(1, n_in + 1, (1,), generator=g))
    return t


def edge_source_table(kvol, n_out, n_in, p, seed):
    """random table whose sources include the first and the last input row in every offset"""
    t = random_table(kvol, n_out, n_in, p, seed)
    g = _gen(seed + 1)
    for k in range(kvol):
        cols = torch.randperm(n_out, generator=g)[:2]
        t[k, cols[0]] = 1
        if n_out > 1:
            t[k, cols[1]] = n_in
    return t


def permute_rows(table, seed):
    """-> (table_p, perm): a random output-row permutation, table_p[:, j] = table[:, perm[j]] (the row_perm contract)"""
    perm = torch.randperm(table.shape[1], generator=_gen(seed)).to(torch.int32)
    return table[:, perm.long()].contiguous(), perm


BUILDERS = ('random', 'empty_tile', 'one_row', 'edge', 'dense')


def build_table(kind, kvol, n_out, n_in, seed):
    if kind == 'random':
        return random_table(kvol, n_out, n_in, 0.4, seed)
    if kind == 'empty_tile':
        return empty_tile_table(kvol, n_out, n_in, 0.5, seed)
    if kind == 'one_row':
        return one_row_per_offset_table(kvol, n_out, n_in, seed)
    if kind == 'edge':
        return edge_source_table(kvol, n_out, n_in, 0.3, seed)
    if kind == 'dense':
        return random_table(kvol, n_out, n_in, 1.0, seed)
    raise ValueError(kind)


# ---- covering design ---------------------------------------------------------------------------------------------------
def pairwise(factors, seed=0, candidates=30):
    """Greedy pairwise covering design: a list of cases (one level per factor, in factor order) in which every pair of
    levels of every two factors occurs at least once.  Deterministic for a seed."""
    rng = random.Random(seed)
    nf = len(factors)
    todo = {(i, a, j, b) for i, j in itertools.combinations(range(nf), 2)
            for a in range(len(factors[i])) for b in range(len(factors[j]))}
    cases = []
    while todo:
        best, best_gain = None, -1
        pool = sorted(todo)
        for _ in range(candidates):
            i0, a0, j0, b0 = rng.choice(pool)  # seed every candidate with one uncovered pair
            case = [None] * nf
            case[i0], case[j0] = a0, b0
            order = [f for f in range(nf) if case[f] is None]
            rng.shuffle(order)
            for f in order:
                gains = []
                for lv in range(len(factors[f])):
                    gain = sum(((min(f, h), lv if f < h else case[h], max(f, h), case[h] if f < h else lv) in todo)
                               for h in range(nf) if case[h] is not None)
                    gains.append(gain)
                top = max(gains)
                case[f] = rng.choice([lv for lv, gv in enumerate(gains) if gv == top])
            gain = sum((i, case[i], j, case[j]) in todo for i, j in itertools.combinations(range(nf), 2))
            if gain > best_gain:
                best, best_gain = case, gain
        for i, j in itertools.combinations(range(nf), 2):
            todo.discard((i, best[i], j, best[j]))
        cases.append(tuple(factors[f][lv] for f, lv in enumerate(best)))
    return cases


def covers_all_pairs(factors, cases):
    for i, j in itertools.combinations(range(len(factors)), 2):
        seen = {(c[i], c[j]) for c in cases}
        if len(seen) != len(factors[i]) * len(factors[j]):
            return False
    return True
