"""Seeded random-input cases for the range coders (the inputs of tests/test_oracle_rans.py's comparisons with the
reference).  Each function runs one case on ANY implementation with the reference's class surface and returns
(summary, streams, inputs): `summary` is what tests/golden/rans_random_golden.json stores (return values, offsets,
CDF tables, stream lengths and SHA-256), `streams` / `inputs` let a caller decode the bytes again."""
import numpy as np

from tests.golden.rans_cases import _h

SIMPLE_SEEDS = (0, 1, 2)


def simple_coder(Encoder, seed):
    rng = np.random.default_rng(seed)
    enc = Encoder(1 << 22)
    calls, rcs = [], []
    for i in range(4):
        n = int(rng.integers(1, 3000))
        S = int(rng.integers(2, 300))
        pm = rng.integers(1, 50, (n, S)) ** 2
        pm = pm * (65536 - S) // pm.sum(1, keepdims=True) + 1
        cdf = np.cumsum(pm, 1); cdf[:, -1] = 65535
        cdf = cdf.astype(np.uint16)
        if i == 2:
            cdf = cdf[:1]
        sym = rng.integers(0, S, n).astype(np.uint16)
        calls.append((cdf, sym))
        rcs.append(enc.encode(cdf, sym))
    stream = bytes(enc.flush())
    return {'encode': rcs, 'stream': _h(stream)}, stream, calls


def indexed_coder(Coder, overflow):
    rng = np.random.default_rng(11)
    T, S, B, n = 7, 20, 3, 2500
    pm = rng.random((T, S)) ** 3 + 1e-4
    pm[1, 10:] = 0
    off = np.full(T, -9, dtype=np.int32)
    coder = Coder(overflow, B)
    coder.init_with_pmfs(pm.copy(), off)
    cdfs = [[int(v) for v in c] for c in coder.get_cdfs()]
    idx = rng.integers(0, T, (B, n)).astype(np.int32)
    if overflow:
        sym = np.round(rng.normal(0, 8, (B, n))).astype(np.int32)
    else:
        lens = np.array([len(c) - 1 for c in cdfs])
        sym = (rng.integers(0, 1 << 30, (B, n)) % lens[idx] + off[idx]).astype(np.int32)
    streams = [bytes(x) for x in coder.encode_with_indexes(sym, idx)]
    return {'offsets': off.tolist(), 'cdfs': cdfs, 'streams': [_h(s) for s in streams]}, streams, (idx, sym)


def binary_coder(Coder):
    rng = np.random.default_rng(3)
    B, n = 2, 30000
    prob = np.clip(np.round(rng.random((B, n)) ** 2 * 65536), 1, 65535).astype(np.uint32)
    sym = rng.random((B, n)) * 65536 < prob
    streams = [bytes(x) for x in Coder(B, 100).encode(sym, prob)]
    return {'streams': [_h(s) for s in streams]}, streams, (prob, sym)


def run_all(RansEncoder, IndexedRansCoder, BinaryRansCoder):
    """-> {case name: summary} for every case, as stored in the golden file"""
    out = {f'simple_{s}': simple_coder(RansEncoder, s)[0] for s in SIMPLE_SEEDS}
    for overflow in (True, False):
        out[f'indexed_overflow_{int(overflow)}'] = indexed_coder(IndexedRansCoder, overflow)[0]
    out['binary'] = binary_coder(BinaryRansCoder)[0]
    return out
