"""Learned entropy model of the latents: the deep-factorized prior with uniform noise, on the device.

Stands in for the reference's lib/entropy_models (continuous_base.py, continuous_batched.py,
distributions/deep_factorized.py, distributions/uniform_noise.py, re-implemented there from tensorflow_compression).
The reference source was not available when this module was written: the definition below is the project's own
(DESIGN 3.10), and neither the constructor signature nor the state-dict keys are a verified drop-in.

  likelihood   L_c(y) = |sigmoid(s f_c(y + 1/2)) - sigmoid(s f_c(y - 1/2))|, f_c the per-channel 1 -> 3 -> 3 -> 3 -> 1
               monotone MLP of DeepFactorized(filters=(3, 3, 3)); bits = -log2(max(L, likelihood_bound))
  training     y + U(-1/2, 1/2) (torch's RNG), bits of the noisy value: one fused kernel each way
               (autograd.FactorizedBitsFunction)
  coding       `update()` samples L on -64 .. 64 per channel (fpcc_factorized_pmf, the same device function), quantises
               the tables with overflow coding (fpcc_pmf_to_quantized_cdf, IndexedRansCoder.init_with_pmfs semantics:
               offset -64, table id = flat index mod C) and keeps them as the module's extra state, so a decoder that
               loads a state dict decodes with the encoder's tables; `compress` / `decompress` run IndexedRansCoder's
               device path on round(y), symbols outside a table through its Elias-gamma escape.

The mean-scale hyperprior (DESIGN 3.11) stands in for the reference's indexed continuous models
(distributions/ noisy normal, continuous_indexed.py, hyperprior/), after compressai's GaussianConditional and Balle et
al.'s mean-scale hyperprior; the same caveat applies (the definition is the project's own, not a verified drop-in).

  likelihood   L = Phi((1/2 - v) / s) - Phi((-1/2 - v) / s), v = |y - mu|, s = max(sigma, scale_bound);
               bits = -log2(max(L, likelihood_bound)), one fused kernel each way (autograd.GaussianBitsFunction)
  coding       `update()` builds one table per entry of the scale table (fpcc_gaussian_pmf, compressai's rule: half-width
               ceil(scale m), m = -Phi^-1(tail_mass / 2)), quantised with overflow coding; each element is coded with
               the table of the smallest scale >= its own (fpcc_gaussian_indexes), in one indexed rANS stream
  hyperprior   z = h_a(y) coded with the deep-factorized prior, (mu, sigma) = h_s(z_hat) conditioning y.  The decoder
               recomputes h_s(z_hat) on the same rows with the same deterministic kernels, so mu, sigma and the table
               indexes are bit-identical on both sides; a decoder on other kernels, another GPU architecture or
               another compute dtype can pick other tables and decode garbage.
"""
import math
from typing import Optional, Tuple

import torch
import torch.nn as nn

from . import _lib, autograd, ops
from . import me as ME
from . import minkowski_sparse_conv_layers as L
from .bitstream import BytesListUtils
from .ops import _p, _s
from .rans_coder import indexed_decode, indexed_encode

PMF_LO, PMF_SYMBOLS = -64, 129
SYMBOL_LIMIT = 1 << 30  # |round(y)| for compress: the escape codes int32 differences to the table


class _CodingTables(nn.Module):
    """quantised CDF tables (cdf_flat int32, cdf_off int64, cdf_len int32, offsets int32) on the device, carried as the
    module's extra state so that a decoder that loads a state dict decodes with the encoder's tables"""

    def _tables_device(self) -> torch.device:
        raise NotImplementedError

    def _quantise(self, pmf, offsets):
        """pmf fp64 [T, S] (consumed), offsets int32 [T] -> tables, with overflow coding (fpcc_pmf_to_quantized_cdf)"""
        T, S = pmf.shape
        cdf = torch.empty((T, S + 2), dtype=torch.int32, device=pmf.device)
        lens = torch.empty(T, dtype=torch.int32, device=pmf.device)
        _lib.call('fpcc_pmf_to_quantized_cdf', _p(pmf), T, S, _p(offsets), 1, _p(cdf), _p(lens), _s())
        if bool((lens < 2).any()):
            raise RuntimeError(f'{type(self).__name__}.update: a table has no symbol to steal frequency from')
        flat = cdf[torch.arange(S + 2, device=cdf.device)[None] < lens[:, None]].contiguous()
        self._set_tables(flat, lens, offsets)

    def _set_tables(self, flat, lens, offsets):
        lens = lens.to(torch.int32).contiguous()
        off = (torch.cumsum(lens.to(torch.int64), 0) - lens).contiguous()
        self._tables = (flat.to(torch.int32).contiguous(), off, lens, offsets.to(torch.int32).contiguous())

    def get_extra_state(self):
        if self._tables is None:
            return {}
        flat, _, lens, offsets = self._tables
        return {'cdf_flat': flat.cpu(), 'cdf_len': lens.cpu(), 'offsets': offsets.cpu()}

    def set_extra_state(self, state):
        if not state:
            self._tables = None
            return
        dev = self._tables_device()
        if dev.type != 'cuda':
            dev = torch.device('cuda', torch.cuda.current_device())
        self._set_tables(state['cdf_flat'].to(dev), state['cdf_len'].to(dev), state['offsets'].to(dev))

    def _need_tables(self, what):
        if self._tables is None:
            raise RuntimeError(f'{type(self).__name__}.{what}: no CDF tables (call update() in eval mode, '
                               'or load a state dict that carries them)')


class NoisyDeepFactorizedEntropyModel(_CodingTables):
    """Per-channel deep-factorized prior of latents y [n, C].

    Parameters (tensorflow_compression's initialisation, scale = init_scale ** (1 / 4)):
      matrices.{i}  [C, d_{i+1}, d_i]  log(expm1(1 / scale / d_{i+1}))     d = (1, 3, 3, 3, 1)
      biases.{i}    [C, d_{i+1}, 1]    U(-1/2, 1/2)
      factors.{i}   [C, d_{i+1}, 1]    0                                    (i < 3)
    forward(y) -> (y_tilde, bits): training, y + U(-1/2, 1/2); eval, round(y) (half to even).  bits fp32 [n, C]."""

    def __init__(self, channels: int, init_scale: float = 10.0, filters=(3, 3, 3), likelihood_bound: float = 1e-9):
        super().__init__()
        if tuple(filters) != (3, 3, 3):
            raise ValueError('NoisyDeepFactorizedEntropyModel: the fused kernels implement filters=(3, 3, 3) only')
        if not 0.0 < likelihood_bound < 1.0:
            raise ValueError('NoisyDeepFactorizedEntropyModel: likelihood_bound must be in (0, 1)')
        self.channels, self.likelihood_bound = int(channels), float(likelihood_bound)
        dims = (1,) + tuple(filters) + (1,)
        scale = init_scale ** (1.0 / (len(filters) + 1))
        self.matrices, self.biases, self.factors = nn.ParameterList(), nn.ParameterList(), nn.ParameterList()
        for i in range(len(filters) + 1):
            init = math.log(math.expm1(1.0 / scale / dims[i + 1]))
            self.matrices.append(nn.Parameter(torch.full((channels, dims[i + 1], dims[i]), init)))
            self.biases.append(nn.Parameter(torch.empty(channels, dims[i + 1], 1).uniform_(-0.5, 0.5)))
            if i < len(filters):
                self.factors.append(nn.Parameter(torch.zeros(channels, dims[i + 1], 1)))
        self._tables = None  # (cdf_flat int32, cdf_off int64, cdf_len int32, offsets int32) on the device

    def params(self) -> torch.Tensor:
        """the packed rows [C, 43] of the kernels: H0 b0 a0 | H1 b1 a1 | H2 b2 a2 | H3 b3 (one torch.cat, so the
        packed gradient flows back to every parameter)"""
        parts = []
        for i in range(4):
            parts += [self.matrices[i].reshape(self.channels, -1), self.biases[i].reshape(self.channels, -1)]
            if i < 3:
                parts.append(self.factors[i].reshape(self.channels, -1))
        return torch.cat(parts, 1).float()

    def forward(self, y: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        yf = y.float()
        if self.training:
            y_q = yf + torch.empty_like(yf).uniform_(-0.5, 0.5)
        else:
            y_q = torch.round(yf)
        bits = autograd.factorized_bits(y_q, self.params(), self.likelihood_bound)
        return y_q.to(y.dtype), bits

    # ---- coding -------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def update(self):
        """builds the quantised CDF tables on the device from the current parameters"""
        if self.training:
            raise RuntimeError('NoisyDeepFactorizedEntropyModel.update: tables are built in eval mode only')
        pmf = ops.factorized_pmf(self.params().detach(), PMF_LO, PMF_SYMBOLS)
        self._quantise(pmf, torch.full((self.channels,), PMF_LO, dtype=torch.int32, device=pmf.device))

    def _tables_device(self):
        return self.matrices[0].device

    @torch.no_grad()
    def compress(self, y: torch.Tensor) -> bytes:
        """y [n, C] (any float dtype, on the device) -> one stream of round(y), table of element (r, c) = c"""
        self._need_tables('compress')
        if y.dim() != 2 or y.shape[1] != self.channels or not y.is_cuda:
            raise RuntimeError(f'NoisyDeepFactorizedEntropyModel.compress: expected a CUDA tensor [n, {self.channels}]')
        if y.shape[0] == 0:
            return b''
        q = torch.round(y.float())
        if not bool((q.abs() < SYMBOL_LIMIT).all()):
            raise RuntimeError('NoisyDeepFactorizedEntropyModel.compress: |round(y)| must be below 2^30')
        sym = q.to(torch.int32).reshape(-1).contiguous()
        return indexed_encode(self._tables, True, sym, None, sym.numel(), 1)[0]

    @torch.no_grad()
    def decompress(self, data: bytes, n: int, device: Optional[torch.device] = None) -> torch.Tensor:
        """-> y_hat fp32 [n, C] on the device"""
        self._need_tables('decompress')
        dev = self._tables[0].device if device is None else torch.device(device)
        if n == 0:
            return torch.empty((0, self.channels), dtype=torch.float32, device=dev)
        blob = torch.frombuffer(bytearray(data) if data else bytearray(1), dtype=torch.uint8).to(dev)
        off = torch.zeros(1, dtype=torch.int64, device=dev)
        ln = torch.tensor([len(data)], dtype=torch.int32, device=dev)
        sym = indexed_decode(self._tables, True, blob, off, ln, None, n * self.channels, 1)
        return sym.reshape(n, self.channels).float()


def default_scale_table() -> torch.Tensor:
    """the 64 log-spaced scales from 0.11 to 256 (compressai's get_scale_table)"""
    return torch.exp(torch.linspace(math.log(0.11), math.log(256.0), 64))


class GaussianConditionalEntropyModel(_CodingTables):
    """Gaussian conditional model of latents y [n, C] given per-element scales and means (compressai's
    GaussianConditional).  scale_table: strictly increasing positive scales, one coding table each (a buffer; default
    `default_scale_table()`).  forward(y, scales, means=None) -> (y_tilde, bits): training, y + U(-1/2, 1/2); eval,
    round(y - mu) + mu (half to even).  bits fp32 [n, C]; gradients reach y, scales and means."""

    def __init__(self, scale_table=None, scale_bound: float = 0.11, tail_mass: float = 1e-9, likelihood_bound: float = 1e-9):
        super().__init__()
        table = default_scale_table() if scale_table is None else torch.as_tensor(scale_table, dtype=torch.float32)
        table = table.float().reshape(-1).clone()
        if table.numel() < 1 or not bool((table > 0).all()) or not bool((table[1:] > table[:-1]).all()):
            raise ValueError('GaussianConditionalEntropyModel: scale_table must be positive and strictly increasing')
        if not 0.0 < scale_bound < float('inf'):
            raise ValueError('GaussianConditionalEntropyModel: scale_bound must be positive')
        if not 0.0 < tail_mass < 1.0 or not 0.0 < likelihood_bound < 1.0:
            raise ValueError('GaussianConditionalEntropyModel: tail_mass and likelihood_bound must be in (0, 1)')
        self.register_buffer('scale_table', table)
        self.scale_bound, self.tail_mass, self.likelihood_bound = float(scale_bound), float(tail_mass), float(likelihood_bound)
        self._tables = None

    def forward(self, y: torch.Tensor, scales: torch.Tensor, means: Optional[torch.Tensor] = None):
        yf = y.float()
        if self.training:
            y_q = yf + torch.empty_like(yf).uniform_(-0.5, 0.5)
        else:
            y_q = torch.round(yf) if means is None else torch.round(yf - means.float()) + means.float()
        bits = autograd.gaussian_bits(y_q, scales, means, self.scale_bound, self.likelihood_bound)
        return y_q.to(y.dtype), bits

    # ---- coding -------------------------------------------------------------------------------------------------
    def _tables_device(self):
        return self.scale_table.device

    @torch.no_grad()
    def update(self):
        """builds one quantised CDF table per scale on the device"""
        if self.training:
            raise RuntimeError('GaussianConditionalEntropyModel.update: tables are built in eval mode only')
        pmf, offsets = ops.gaussian_pmf(self.scale_table, self.tail_mass)
        self._quantise(pmf, offsets)

    def _rows(self, t, n, C, what):
        if t is None:
            return None
        if t.dim() != 2 or tuple(t.shape) != (n, C) or not t.is_cuda:
            raise RuntimeError(f'GaussianConditionalEntropyModel.{what}: expected CUDA tensors [n, C] of one shape')
        return t.float()

    @torch.no_grad()
    def compress(self, y: torch.Tensor, scales: torch.Tensor, means: Optional[torch.Tensor] = None) -> bytes:
        """y, scales, means [n, C] on the device -> one stream of round(y - mu), element (r, c) coded with the table
        of the smallest scale >= max(scales[r, c], scale_bound)"""
        self._need_tables('compress')
        n, C = y.shape if y.dim() == 2 else (-1, -1)
        yf, s, m = self._rows(y, n, C, 'compress'), self._rows(scales, n, C, 'compress'), self._rows(means, n, C, 'compress')
        if n == 0 or C == 0:
            return b''
        d = yf if m is None else yf - m
        if not bool((d.abs() < SYMBOL_LIMIT).all()):
            raise RuntimeError('GaussianConditionalEntropyModel.compress: |round(y - mu)| must be below 2^30')
        sym, idx = ops.gaussian_indexes(self.scale_table, s, m, yf, self.scale_bound)
        return indexed_encode(self._tables, True, sym.reshape(-1), idx.reshape(-1), n * C, 1)[0]

    @torch.no_grad()
    def decompress(self, data: bytes, scales: torch.Tensor, means: Optional[torch.Tensor] = None) -> torch.Tensor:
        """-> y_hat fp32 [n, C] = decoded symbols + mu, with the scales and means of the encoder"""
        self._need_tables('decompress')
        n, C = scales.shape if scales.dim() == 2 else (-1, -1)
        s, m = self._rows(scales, n, C, 'decompress'), self._rows(means, n, C, 'decompress')
        if n == 0 or C == 0:
            return torch.empty((n, C), dtype=torch.float32, device=s.device)
        idx = ops.gaussian_indexes(self.scale_table, s, None, None, self.scale_bound)
        blob = torch.frombuffer(bytearray(data) if data else bytearray(1), dtype=torch.uint8).to(s.device)
        off = torch.zeros(1, dtype=torch.int64, device=s.device)
        ln = torch.tensor([len(data)], dtype=torch.int32, device=s.device)
        sym = indexed_decode(self._tables, True, blob, off, ln, idx.reshape(-1), n * C, 1).reshape(n, C).float()
        return sym if m is None else sym + m


class HyperpriorEntropyModel(nn.Module):
    """Mean-scale hyperprior on MinkowskiEngine-shim sparse tensors (Balle et al. / Minnen et al., as compressai builds
    it), for latents y of `latent` channels at any tensor stride ts:

      h_a   ConvBlock(latent -> hyper_channels, k2 s2) -> MEMLPBlock(hyper_channels -> hyper_latent, no act)    z, stride 2 ts
      z     NoisyDeepFactorizedEntropyModel(hyper_latent)
      h_s   ConvTransBlock(hyper_latent -> hyper_channels, k2 s2) onto y's coordinate key
            -> MEMLPBlock(hyper_channels -> 2 latent, no act) = (mu, sigma), the two column halves
      y     GaussianConditionalEntropyModel, given (mu, sigma)

    forward(y) -> (y_tilde SparseTensor on y's key, bits_y fp32 [n_y, latent], bits_z fp32 [n_z, hyper_latent]).
    compress(y) -> bytes (the z stream and the y stream joined with BytesListUtils); decompress(data, y_skeleton) takes
    a tensor that carries only y's coordinates (any features) and rebuilds z's coordinates with
    CoordinateManager.stride, as h_a's conv does.  Decoding needs mu and sigma bit-identical to the encoder's: the
    same kernels on the same rows in the same compute dtype (see the module docstring)."""

    def __init__(self, latent: int, hyper_latent: int, hyper_channels: int):
        super().__init__()
        self.latent = int(latent)
        self.h_a_conv = L.ConvBlock(latent, hyper_channels, 2, 2)
        self.h_a_mlp = L.MEMLPBlock(hyper_channels, hyper_latent, act=None)
        self.h_s_conv = L.ConvTransBlock(hyper_latent, hyper_channels, 2, 2)
        self.h_s_mlp = L.MEMLPBlock(hyper_channels, 2 * latent, act=None)
        self.hyper_prior = NoisyDeepFactorizedEntropyModel(hyper_latent)
        self.conditional = GaussianConditionalEntropyModel()

    def means_scales(self, z_hat, y_key):
        """h_s(z_hat) onto y's key -> (mu, sigma), fp32 column halves of one [n_y, 2 latent] tensor"""
        ms = self.h_s_mlp(self.h_s_conv(z_hat, y_key)).F.float()
        return ms[:, :self.latent], ms[:, self.latent:]

    def forward(self, y):
        z = self.h_a_mlp(self.h_a_conv(y))
        z_t, bits_z = self.hyper_prior(z.F)
        mu, sigma = self.means_scales(z._like(z_t), y.coordinate_map_key)
        y_t, bits_y = self.conditional(y.F, sigma, mu)
        return y._like(y_t), bits_y, bits_z

    @torch.no_grad()
    def update(self):
        self.hyper_prior.update()
        self.conditional.update()

    @torch.no_grad()
    def compress(self, y) -> bytes:
        z = self.h_a_mlp(self.h_a_conv(y))
        z_data = self.hyper_prior.compress(z.F)
        z_hat = torch.round(z.F.float()).to(z.F.dtype)          # what the decoder gets back, in the same dtype
        mu, sigma = self.means_scales(z._like(z_hat), y.coordinate_map_key)
        y_data = self.conditional.compress(y.F, sigma, mu)
        return BytesListUtils.concat_bytes_list([z_data, y_data])

    @torch.no_grad()
    def decompress(self, data: bytes, y_skeleton):
        """-> y_hat SparseTensor on y_skeleton's key, fp32 features [n_y, latent]"""
        z_data, y_data = BytesListUtils.split_bytes_list(data, 2)
        cm, y_key = y_skeleton.coordinate_manager, y_skeleton.coordinate_map_key
        z_key = cm.stride(y_key, 2)
        n_z = cm.get_coordinates(z_key).shape[0]
        z_hat = self.hyper_prior.decompress(z_data, n_z, device=cm.get_coordinates(y_key).device)
        z_hat = ME.SparseTensor(z_hat.to(ME.compute_dtype()), coordinate_map_key=z_key, coordinate_manager=cm)
        mu, sigma = self.means_scales(z_hat, y_key)
        return ME.SparseTensor(self.conditional.decompress(y_data, sigma, mu), coordinate_map_key=y_key, coordinate_manager=cm)
