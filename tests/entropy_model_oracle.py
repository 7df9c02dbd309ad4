"""Float64 torch restatement of the deep-factorized entropy model (DESIGN 3.10; csrc/entropy_model.cu): the forward
f_c, the likelihood with its sign choice, the bounded bits with compressai's LowerBound gradient rule, written with
plain tensor ops so that torch autograd gives the reference dy and dparams of fpcc_factorized_grad."""
import torch

NP = 43


def unpack(params: torch.Tensor):
    """[C, 43] -> per layer (H [C, out, in], b [C, out], a [C, out] | None)"""
    C = params.shape[0]
    shapes = [(3, 1), (3, 3), (3, 3), (1, 3)]
    out, o = [], 0
    for i, (r, c) in enumerate(shapes):
        H = params[:, o:o + r * c].reshape(C, r, c)
        o += r * c
        b = params[:, o:o + r]
        o += r
        a = None
        if i < 3:
            a = params[:, o:o + r]
            o += r
        out.append((H, b, a))
    assert o == NP
    return out


def logits(params: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    """f_c(x) for x [n, C] -> [n, C]"""
    v = x[..., None]  # [n, C, 1]
    for H, b, a in unpack(params):
        v = torch.einsum('coi,nci->nco', torch.nn.functional.softplus(H), v) + b[None]
        if a is not None:
            v = v + torch.tanh(a)[None] * torch.tanh(v)
    return v[..., 0]


def likelihood(params: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
    u, l = logits(params, y + 0.5), logits(params, y - 0.5)
    s = torch.where(u + l > 0, -torch.ones_like(u), torch.ones_like(u))
    return (torch.sigmoid(s * u) - torch.sigmoid(s * l)).abs()


class LowerBound(torch.autograd.Function):
    """max(x, bound); the gradient passes where x >= bound or where it would raise x (compressai's LowerBound)"""

    @staticmethod
    def forward(ctx, x, bound):
        ctx.save_for_backward(x)
        ctx.bound = bound
        return x.clamp(min=bound)

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        return g * ((x >= ctx.bound) | (g < 0)).to(g.dtype), None


def bits(params: torch.Tensor, y: torch.Tensor, bound: float = 1e-9) -> torch.Tensor:
    return -torch.log2(LowerBound.apply(likelihood(params, y), bound))


def random_params(C: int, gen: torch.Generator, spread: float = 1.0) -> torch.Tensor:
    """params [C, 43] fp64 around the initialisation of NoisyDeepFactorizedEntropyModel (init_scale 10) with noise"""
    import math
    scale = 10.0 ** 0.25
    base = torch.zeros(NP, dtype=torch.float64)
    o = 0
    for i, (r, c) in enumerate([(3, 1), (3, 3), (3, 3), (1, 3)]):
        base[o:o + r * c] = math.log(math.expm1(1.0 / scale / r))
        o += r * c + r + (r if i < 3 else 0)
    return base[None] + spread * torch.randn((C, NP), dtype=torch.float64, generator=gen)
