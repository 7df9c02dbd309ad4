"""Mints tests/golden/rans_random_golden.json: the outputs of the range coders on the seeded random inputs of
tests/golden/rans_random_cases.py.

    python tests/golden/make_rans_random_golden.py

The vectors are those of the C restatement (oracle/rans_oracle.c).  When the reference's own coders are built
(oracle/_ref, see oracle/build_ref.py) they are run on the same inputs and must give identical outputs, or nothing
is written.  The file in the repository was minted from the C restatement as it was when it was pinned byte for byte
against the compiled reference on exactly these inputs (the restatement, its ctypes front-end and these inputs have not
changed since); tests/test_oracle_rans.py checks the vectors against the reference again wherever it is built.
"""
import json
import os.path as osp
import sys

import numpy as np

ROOT = osp.dirname(osp.dirname(osp.dirname(osp.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import build_ref  # noqa: E402
from oracle import rans as orans  # noqa: E402
from tests.golden import rans_random_cases  # noqa: E402


def main():
    out = rans_random_cases.run_all(orans.RansEncoder, orans.IndexedRansCoder, orans.BinaryRansCoder)
    simple, batched = build_ref.load_ref('simple_rans_ext_cpp'), build_ref.load_ref('rans_ext_cpp')
    checked = simple is not None and batched is not None
    if checked:
        ref = rans_random_cases.run_all(simple.RansEncoder, batched.IndexedRansCoder, batched.BinaryRansCoder)
        assert ref == out, 'the C restatement differs from the reference coders'
    out['_meta'] = {'minted_from': 'oracle/rans_oracle.c' + (', equal to the reference coders (oracle/_ref)' if checked else ''),
                    'numpy': np.__version__}
    with open(osp.join(osp.dirname(osp.abspath(__file__)), 'rans_random_golden.json'), 'w') as f:
        json.dump(out, f, indent=1, sort_keys=True)
    for k, v in out.items():
        print(k, str(v)[:100])


if __name__ == '__main__':
    main()
