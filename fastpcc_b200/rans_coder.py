"""GPU range coders with the reference's Python class surface (numpy in, bytes out):

  RansEncoder / RansDecoder ...... models/convolutional/lossy_coord_v3/rans_coder (simple_rans_wrapper.cpp:272-286)
  IndexedRansCoder, BinaryRansCoder,
  batched_pmf_to_quantized_cdf ... lib/entropy_models/rans_coder (rans_wrapper.cpp:430-451)

Bitstreams are byte-identical to the reference's CPU coders.  These classes are the drop-in boundary; the
codec models call the device-resident entry points in `ops` directly and never round-trip through numpy.
"""
from typing import List

import numpy as np
import torch

from . import _lib, ops
from .ops import _p, _s


def _dev(a, dtype=None):
    t = torch.from_numpy(np.array(a, copy=True, order='C'))
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda()


class RansEncoder:
    def __init__(self, enc_buf_size: int = 32 * 1024 * 1024):
        assert enc_buf_size > 0
        self._cap = int(enc_buf_size)
        self._buf = None
        self._state = None

    def _ensure(self):
        if self._buf is None:
            self._buf = torch.empty((1, self._cap), dtype=torch.uint8, device='cuda')
            self._state = torch.tensor([[1 << 23, 0]], dtype=torch.int32, device='cuda')

    def _push(self, ranges, flush):
        self._ensure()
        n = 0 if ranges is None else ranges.numel()
        if ranges is None:
            ranges = torch.empty(1, dtype=torch.int32, device='cuda')
        off = torch.tensor([0, n], dtype=torch.int64, device='cuda')
        _, out_len = ops.rans_encode(ranges, off, self._cap, out=self._buf, state_io=self._state, flush=flush, total=n)
        size = int(out_len.item())
        if size < 0:
            raise RuntimeError('RansEncoder: enc_buf_size exceeded')
        return size

    def encode(self, cdf_arr: np.ndarray, symbol_arr: np.ndarray) -> int:
        """simple_rans_wrapper.cpp:67-95: cdf uint16 [n,S] (or [1,S] shared), symbols uint16 [n]."""
        assert cdf_arr.dtype == np.uint16 and cdf_arr.ndim == 2 and symbol_arr.dtype == np.uint16
        assert cdf_arr.shape[0] in (1, symbol_arr.shape[0])
        if symbol_arr.shape[0] == 0:
            return self._push(None, False)
        ranges = ops.table_symbol_ranges(_dev(cdf_arr), _dev(symbol_arr.astype(np.int32)))
        return self._push(ranges, False)

    def encode_bin(self, cdf_arr: np.ndarray, symbol_arr: np.ndarray) -> int:
        """simple_rans_wrapper.cpp:97-124: a [n] (or [1]) threshold table = two-symbol CDF rows."""
        thr = np.ascontiguousarray(cdf_arr, dtype=np.uint16).reshape(-1, 1)
        rows = np.concatenate([thr, np.full_like(thr, 65535)], 1)
        return self.encode(rows, np.ascontiguousarray(symbol_arr).astype(np.uint16))

    def flush(self) -> bytes:
        size = self._push(None, True)
        data = self._buf[0, self._cap - size:].cpu().numpy().tobytes()
        self._state = torch.tensor([[1 << 23, 0]], dtype=torch.int32, device='cuda')
        return data


class RansDecoder:
    def __init__(self):
        self._dec = None

    def flush(self, encoded: bytes) -> int:
        data = torch.frombuffer(bytearray(encoded), dtype=torch.uint8).cuda()
        self._dec = ops.RansDecodeStreams(data, torch.zeros(1, dtype=torch.int64, device='cuda'),
                                          torch.tensor([len(encoded)], dtype=torch.int32, device='cuda'))
        return 0

    def decode(self, cdf_arr: np.ndarray, symbol_arr: np.ndarray) -> int:
        """simple_rans_wrapper.cpp:206-239: fills symbol_arr in place."""
        assert cdf_arr.dtype == np.uint16 and cdf_arr.ndim == 2 and symbol_arr.dtype == np.uint16
        n = symbol_arr.shape[0]
        assert cdf_arr.shape[0] in (1, n)
        if n == 0:
            return 0
        row_off = torch.tensor([0, n], dtype=torch.int64, device='cuda')
        sym = self._dec.decode(_dev(cdf_arr), cdf_arr.shape[1], row_off, n, shared=cdf_arr.shape[0] == 1 and n != 1)
        symbol_arr[...] = sym.cpu().numpy().astype(np.uint16)
        if self._dec.error():
            raise RuntimeError('RansDecoder: read past the end of the stream')
        return 0

    def decode_bin(self, cdf_arr: np.ndarray, symbol_arr: np.ndarray) -> int:
        thr = np.ascontiguousarray(cdf_arr, dtype=np.uint16).reshape(-1, 1)
        rows = np.concatenate([thr, np.full_like(thr, 65535)], 1)
        tmp = np.empty(symbol_arr.shape[0], dtype=np.uint16)
        self.decode(rows, tmp)
        symbol_arr[...] = tmp.astype(np.bool_)
        return 0


def batched_pmf_to_quantized_cdf(pmf_array: np.ndarray, offset_array: np.ndarray, overflow_coding: bool) -> List[List[int]]:
    """cdf_ops.cpp:111-143 on the GPU (one thread per table, fp64 in the reference's evaluation order).
    `offset_array` is adjusted in place in overflow mode and `pmf_array` becomes its prefix sums."""
    assert pmf_array.dtype == np.float64 and pmf_array.ndim == 2 and offset_array.dtype == np.int32
    T, S = pmf_array.shape
    d_pmf, d_off = _dev(pmf_array), _dev(offset_array)
    cdf = torch.empty((T, S + 2), dtype=torch.int32, device='cuda')
    lens = torch.empty(T, dtype=torch.int32, device='cuda')
    _lib.call('fpcc_pmf_to_quantized_cdf', _p(d_pmf), T, S, _p(d_off), int(bool(overflow_coding)), _p(cdf), _p(lens), _s())
    lens_h = lens.cpu().numpy()
    if (lens_h < 0).any():
        raise RuntimeError('pmf_to_quantized_cdf: no symbol to steal frequency from')
    cdf_h = cdf.cpu().numpy().view(np.uint32)
    pmf_array[...] = d_pmf.cpu().numpy()
    offset_array[...] = d_off.cpu().numpy()
    return [cdf_h[t, :lens_h[t]].tolist() for t in range(T)]


def _table_args(tables, overflow):
    flat, off, lens, offsets = tables
    return _p(flat), _p(off), _p(lens), lens.numel(), _p(offsets), int(bool(overflow))


def indexed_encode(tables, overflow, sym, idx, n, n_streams):
    """IndexedRansCoder's encoder on device tensors: tables = (cdf_flat int32, cdf_off int64, cdf_len int32, offsets
    int32), sym int32 [n_streams * n] (idx: int32 table ids, or None for table = position mod n_tables)
    -> one bytes object per stream"""
    cnt = torch.empty(n_streams * n, dtype=torch.int32, device=sym.device)
    _lib.call('fpcc_indexed_count', *_table_args(tables, overflow), _p(sym), _p(idx), n, n_streams, _p(cnt), _s())
    incl = torch.cumsum(cnt.to(torch.int64), 0)
    pos = (incl - cnt).contiguous()
    total = int(incl[-1].item())
    ranges = torch.empty(total, dtype=torch.int32, device=sym.device)
    bits = torch.empty(total, dtype=torch.uint8, device=sym.device)
    _lib.call('fpcc_indexed_ranges', *_table_args(tables, overflow), _p(sym), _p(idx), n, n_streams, _p(pos), _p(ranges), _p(bits), _s())
    rng_off = torch.cat([pos[::n], incl[-1:]]).contiguous()
    per = (rng_off[1:] - rng_off[:-1])
    cap = int(per.max().item()) * 2 + 64
    out, out_len = ops.rans_encode(ranges, rng_off, cap, bits=bits)
    out, out_len = out.cpu().numpy(), out_len.cpu().numpy()
    assert (out_len > 0).all()
    return [out[b, cap - out_len[b]:].tobytes() for b in range(n_streams)]


def indexed_decode(tables, overflow, blob, byte_off, byte_len, idx, n, n_streams):
    """IndexedRansCoder's decoder on device tensors (streams at blob[byte_off[b]:][:byte_len[b]]) -> int32 [n_streams, n]
    on the device; raises when a stream ends early"""
    out = torch.empty((n_streams, n), dtype=torch.int32, device=blob.device)
    err = torch.zeros(1, dtype=torch.int32, device=blob.device)
    _lib.call('fpcc_indexed_decode', *_table_args(tables, overflow), _p(blob), _p(byte_off), _p(byte_len), _p(idx), n, n_streams,
              _p(out), _p(err), _s())
    if int(err.item()):
        raise RuntimeError('IndexedRansCoder: read past the end of a stream')
    return out


class IndexedRansCoder:
    def __init__(self, overflow_coding: bool, batch_size: int, enc_buf_size: int = 8 * 1024 * 1024):
        assert batch_size > 0
        self.overflow_coding, self.batch_size = bool(overflow_coding), int(batch_size)
        self.cdfs = None
        self.offset_array = None

    def init_with_pmfs(self, pmf_array, offset_array):
        return self.init_with_quantized_cdfs(batched_pmf_to_quantized_cdf(pmf_array, offset_array, self.overflow_coding), offset_array)

    def init_with_quantized_cdfs(self, cdfs, offset_array):
        self.cdfs = [list(map(int, c)) for c in cdfs]
        self.offset_array = offset_array
        lens = np.array([len(c) for c in self.cdfs], dtype=np.int32)
        self._t = (_dev(np.concatenate([np.asarray(c, dtype=np.uint32) for c in self.cdfs]).view(np.int32)),
                   _dev(np.concatenate([[0], np.cumsum(lens[:-1])]).astype(np.int64)), _dev(lens),
                   _dev(np.ascontiguousarray(offset_array, dtype=np.int32)))
        return 0

    def get_cdfs(self):
        return self.cdfs

    def get_offset_array(self):
        return self.offset_array

    def _encode(self, symbol_array, index_array):
        sym = np.ascontiguousarray(symbol_array, dtype=np.int32)
        assert sym.ndim == 2 and sym.shape[0] == self.batch_size
        B, n = sym.shape
        d_sym = _dev(sym)
        d_idx = _dev(np.ascontiguousarray(index_array, dtype=np.int32)) if index_array is not None else None
        return indexed_encode(self._t, self.overflow_coding, d_sym, d_idx, n, B)

    def encode(self, symbol_array):
        return self._encode(symbol_array, None)

    def encode_with_indexes(self, symbol_array, index_array):
        return self._encode(symbol_array, index_array)

    def _decode(self, encoded_list, index_array, symbol_array):
        assert symbol_array.dtype == np.int32 and symbol_array.ndim == 2 and len(encoded_list) == self.batch_size
        B, n = symbol_array.shape
        blob = np.frombuffer(b''.join(bytes(e) for e in encoded_list), dtype=np.uint8)
        lens = np.array([len(e) for e in encoded_list], dtype=np.int32)
        d_idx = _dev(np.ascontiguousarray(index_array, dtype=np.int32)) if index_array is not None else None
        d_blob, d_off, d_len = _dev(blob), _dev(np.concatenate([[0], np.cumsum(lens[:-1])]).astype(np.int64)), _dev(lens)
        symbol_array[...] = indexed_decode(self._t, self.overflow_coding, d_blob, d_off, d_len, d_idx, n, B).cpu().numpy()
        return 0

    def decode(self, encoded_list, symbol_array):
        return self._decode(encoded_list, None, symbol_array)

    def decode_with_indexes(self, encoded_list, index_array, symbol_array):
        return self._decode(encoded_list, index_array, symbol_array)


class BinaryRansCoder:
    def __init__(self, batch_size: int, enc_buf_size: int = 8 * 1024 * 1024):
        assert batch_size > 0
        self.batch_size = int(batch_size)

    def encode(self, symbol_array, prob_array):
        """rans_wrapper.cpp:326-382: symbols bool [B,n], prob uint32 [B,n] = P(1)*65536 in [1,65535]."""
        sym = np.ascontiguousarray(symbol_array, dtype=np.bool_).view(np.uint8)
        prob = np.ascontiguousarray(prob_array, dtype=np.uint32)
        assert sym.ndim == 2 and sym.shape == prob.shape and sym.shape[0] == self.batch_size
        B, n = sym.shape
        ranges = torch.empty(B * n, dtype=torch.int32, device='cuda')
        d_sym, d_prob = _dev(sym), _dev(prob.view(np.int32))  # named: both must stay alive until the launch
        _lib.call('fpcc_rans_binary_ranges', _p(d_sym), _p(d_prob), B * n, _p(ranges), _s())
        rng_off = torch.arange(0, (B + 1) * n, n, dtype=torch.int64, device='cuda')
        cap = 2 * n + 64
        out, out_len = ops.rans_encode(ranges, rng_off, cap)
        out, out_len = out.cpu().numpy(), out_len.cpu().numpy()
        assert (out_len > 0).all()
        return [out[b, cap - out_len[b]:].tobytes() for b in range(B)]

    def decode(self, encoded_list, prob_array, symbol_array):
        prob = np.ascontiguousarray(prob_array, dtype=np.uint32)
        assert symbol_array.dtype == np.bool_ and symbol_array.shape == prob.shape and len(encoded_list) == self.batch_size
        B, n = prob.shape
        blob = np.frombuffer(b''.join(bytes(e) for e in encoded_list), dtype=np.uint8)
        lens = np.array([len(e) for e in encoded_list], dtype=np.int32)
        out = torch.empty((B, n), dtype=torch.uint8, device='cuda')
        err = torch.zeros(1, dtype=torch.int32, device='cuda')
        d_blob, d_off, d_len = _dev(blob), _dev(np.concatenate([[0], np.cumsum(lens[:-1])]).astype(np.int64)), _dev(lens)
        d_prob = _dev(prob.view(np.int32))
        _lib.call('fpcc_rans_binary_decode', _p(d_blob), _p(d_off), _p(d_len), _p(d_prob), n, B, _p(out), _p(err), _s())
        symbol_array[...] = out.cpu().numpy().astype(np.bool_)
        if int(err.item()):
            raise RuntimeError('BinaryRansCoder: read past the end of a stream')
        return 0
