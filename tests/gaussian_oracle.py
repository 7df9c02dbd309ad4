"""Float64 torch restatement of the Gaussian conditional entropy model (DESIGN 3.11; csrc/entropy_model.cu): the
likelihood with torch.special.erfc, both lower bounds with compressai's LowerBound gradient rule, the table rule and the
index rule, written with plain tensor ops so that torch autograd gives the reference dy, dmu and dsigma of
fpcc_gaussian_grad."""
import math

import torch

from tests.entropy_model_oracle import LowerBound


def cdf(x: torch.Tensor) -> torch.Tensor:
    """Phi(x) = erfc(-x / sqrt 2) / 2"""
    return 0.5 * torch.special.erfc(-x / math.sqrt(2.0))


def likelihood(y, scales, means=None, scale_bound=0.11):
    v = (y if means is None else y - means).abs()
    s = LowerBound.apply(scales, scale_bound)
    return cdf((0.5 - v) / s) - cdf((-0.5 - v) / s)


def bits(y, scales, means=None, scale_bound=0.11, bound=1e-9):
    return -torch.log2(LowerBound.apply(likelihood(y, scales, means, scale_bound), bound))


def tail_multiplier(tail_mass=1e-9) -> float:
    """m = -Phi^-1(tail_mass / 2)"""
    return -float(torch.special.ndtri(torch.tensor(tail_mass / 2, dtype=torch.float64)))


def pmf_rows(scale_table, centers):
    """pmf fp64 [T, 2 max(center) + 1]: row t = L(k) at mean 0 and sigma = scale_table[t] (unbounded) for
    k = -center_t .. center_t, zero beyond"""
    T, S = len(centers), 2 * int(max(centers)) + 1
    pmf = torch.zeros((T, S), dtype=torch.float64)
    for t, c in enumerate(centers):
        k = torch.arange(-c, c + 1, dtype=torch.float64)
        s = float(scale_table[t])
        pmf[t, :2 * c + 1] = cdf((0.5 - k.abs()) / s) - cdf((-0.5 - k.abs()) / s)
    return pmf


def indexes(scales, scale_table, scale_bound=0.11):
    """compressai's build_indexes: T - 1 minus the number of table entries t < T - 1 with max(sigma, bound) <= table[t]"""
    s = scales.clamp(min=scale_bound)
    idx = torch.full(s.shape, len(scale_table) - 1, dtype=torch.int64)
    for t in scale_table[:-1]:
        idx -= (s <= t).to(torch.int64)
    return idx
