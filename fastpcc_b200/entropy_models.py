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
"""
import math
from typing import Optional, Tuple

import torch
import torch.nn as nn

from . import _lib, autograd, ops
from .ops import _p, _s
from .rans_coder import indexed_decode, indexed_encode

PMF_LO, PMF_SYMBOLS = -64, 129
SYMBOL_LIMIT = 1 << 30  # |round(y)| for compress: the escape codes int32 differences to the table


class NoisyDeepFactorizedEntropyModel(nn.Module):
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
        params = self.params().detach()
        C = self.channels
        pmf = ops.factorized_pmf(params, PMF_LO, PMF_SYMBOLS)
        offsets = torch.full((C,), PMF_LO, dtype=torch.int32, device=pmf.device)
        cdf = torch.empty((C, PMF_SYMBOLS + 2), dtype=torch.int32, device=pmf.device)
        lens = torch.empty(C, dtype=torch.int32, device=pmf.device)
        _lib.call('fpcc_pmf_to_quantized_cdf', _p(pmf), C, PMF_SYMBOLS, _p(offsets), 1, _p(cdf), _p(lens), _s())
        if bool((lens < 2).any()):
            raise RuntimeError('NoisyDeepFactorizedEntropyModel.update: a table has no symbol to steal frequency from')
        flat = cdf[torch.arange(PMF_SYMBOLS + 2, device=cdf.device)[None] < lens[:, None]].contiguous()
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
        dev = self.matrices[0].device
        if dev.type != 'cuda':
            dev = torch.device('cuda', torch.cuda.current_device())
        self._set_tables(state['cdf_flat'].to(dev), state['cdf_len'].to(dev), state['offsets'].to(dev))

    def _need_tables(self, what):
        if self._tables is None:
            raise RuntimeError(f'NoisyDeepFactorizedEntropyModel.{what}: no CDF tables (call update() in eval mode, '
                               'or load a state dict that carries them)')

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
