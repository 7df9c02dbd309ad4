"""The float oracle of the lossy codec is deterministic and matches its committed fixture: the reference's unmodified
lossy_coord_v2 model (imported from $FASTPCC_REFERENCE_ROOT, or from the staged oracle/_ref/pyref.zip) on the CPU
MinkowskiEngine stand-in (oracle/me_cpu.py) reproduces tests/golden/lossy_v2_golden.json -- bytes, decoded point count,
D1 PSNR and the losslessly coded stride-2 geometry."""
import json
import os.path as osp
import zipfile

import numpy as np
import pytest

ROOT = osp.dirname(osp.dirname(osp.abspath(__file__)))
PYREF = osp.join(ROOT, 'oracle', '_ref', 'pyref.zip')


def reference_root(tmp_path_factory):
    from oracle import build_ref
    if build_ref.REF_ROOT and osp.isdir(osp.join(build_ref.REF_ROOT, 'models')):
        return build_ref.REF_ROOT
    if osp.isfile(PYREF):
        root = str(tmp_path_factory.mktemp('pyref'))
        with zipfile.ZipFile(PYREF) as z:
            z.extractall(root)
        return root
    pytest.skip('reference Python not staged (set FASTPCC_REFERENCE_ROOT to a checkout of the reference, or run oracle/build_ref.py there)')


def golden():
    return {g['name']: g for g in json.load(open(osp.join(ROOT, 'tests', 'golden', 'lossy_v2_golden.json')))['cases']}


@pytest.mark.timeout(600)
def test_reference_lossy_v2_on_the_cpu_oracle_matches_its_fixture(tmp_path_factory):
    from oracle import build_ref, me_cpu, metrics
    from tests import ref_import
    from tests.golden.lossy_cases import CASES
    from tests.golden.make_lossy_golden import run_case, stride2_sha
    rans = build_ref.load_ref('rans_ext_cpp')
    if rans is None:
        pytest.skip('oracle/_ref/rans_ext_cpp not built')
    me = me_cpu.load('MinkowskiEngine_cpu_oracle')
    ref = ref_import.import_reference_lossy_v2(reference_root(tmp_path_factory), me, rans=rans)
    case = [c for c in CASES if c['name'] == 'v2_r1_6k'][0]
    g = golden()[case['name']]
    xyz, data, rec = run_case(ref, case)
    assert len(data) == g['n_bytes'] and rec.shape[0] == g['n_rec'] == xyz.shape[0]
    err = metrics.pc_error(xyz, rec, 2 ** case['bits'])
    assert abs(err['mseF,PSNR (p2point)'] - g['d1_psnr']) < 1e-9
    # the entropy model codes the stride-2 geometry losslessly, and the top-k pruning keeps the best child of every cell
    assert stride2_sha(rec, xyz.min(0))[0] == g['stride2_sha256'] == stride2_sha(xyz, xyz.min(0))[0]
