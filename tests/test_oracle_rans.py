"""Pins the C restatement of the range coders (oracle/rans_oracle.c):
(1) against the committed golden vectors minted from the compiled reference, and
(2) byte-for-byte against the reference's outputs on seeded random inputs: the committed vectors of
tests/golden/rans_random_golden.json, and the compiled reference itself (oracle/_ref) when it is built."""
import json
import os.path as osp

import numpy as np
import pytest

from oracle import rans as orans
from oracle import build_ref
from tests.golden import rans_cases, rans_random_cases as R

with open(osp.join(osp.dirname(__file__), 'golden', 'rans_random_golden.json')) as _f:
    RANDOM_GOLDEN = json.load(_f)


def test_oracle_matches_golden(rans_kat):
    got = rans_cases.run_all(orans.RansEncoder, orans.RansDecoder, orans.IndexedRansCoder,
                             orans.BinaryRansCoder, orans.batched_pmf_to_quantized_cdf)
    for k, v in rans_kat.items():
        if k.startswith('_'):
            continue
        assert got[k] == v, k


def _ref():
    """-> (simple_rans_ext_cpp, rans_ext_cpp), the reference's compiled coders, or None when they are not built"""
    s = build_ref.load_ref('simple_rans_ext_cpp')
    b = build_ref.load_ref('rans_ext_cpp')
    return (s, b) if s is not None and b is not None else None


@pytest.mark.parametrize('seed', R.SIMPLE_SEEDS)
def test_simple_coder_vs_reference(seed):
    got, stream, calls = R.simple_coder(orans.RansEncoder, seed)
    assert got == RANDOM_GOLDEN[f'simple_{seed}']
    ref = _ref()
    if ref is not None:
        assert R.simple_coder(ref[0].RansEncoder, seed)[0] == got
    decoders = [orans.RansDecoder()] + ([ref[0].RansDecoder()] if ref is not None else [])
    for dec in decoders:
        dec.flush(stream)
    for cdf, sym in reversed(calls):
        for dec in decoders:
            out = np.zeros_like(sym)
            dec.decode(cdf, out)
            assert (out == sym).all()


@pytest.mark.parametrize('overflow', [True, False])
def test_indexed_coder_vs_reference(overflow):
    got, streams, (idx, sym) = R.indexed_coder(orans.IndexedRansCoder, overflow)
    assert got == RANDOM_GOLDEN[f'indexed_overflow_{int(overflow)}']
    ref = _ref()
    if ref is not None:
        assert R.indexed_coder(ref[1].IndexedRansCoder, overflow)[0] == got
    co = orans.IndexedRansCoder(overflow, idx.shape[0])
    co.init_with_quantized_cdfs(got['cdfs'], np.array(got['offsets'], dtype=np.int32))
    d = np.empty_like(sym)
    co.decode_with_indexes(streams, idx, d)
    assert (d == sym).all()


def test_binary_coder_vs_reference():
    got, streams, (prob, sym) = R.binary_coder(orans.BinaryRansCoder)
    assert got == RANDOM_GOLDEN['binary']
    ref = _ref()
    if ref is not None:
        assert R.binary_coder(ref[1].BinaryRansCoder)[0] == got
    d = np.empty_like(sym)
    orans.BinaryRansCoder(sym.shape[0]).decode(streams, prob, d)
    assert (d == sym).all()
