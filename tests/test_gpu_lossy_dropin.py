"""The float drop-in boundary on the GPU: the reference's OWN, UNMODIFIED lossy object codec
(models/convolutional/lossy_coord_v2/model.py:230-275 PCC.compress / decompress, layers.py Encoder / Decoder with
top-k pruning, lossy_coord_lossy_color/geo_lossl_em.py GeoLosslessEntropyModel, lib/minkowski_sparse_conv_layers.py)
runs with

    MinkowskiEngine              :=  fastpcc_b200.me          (fp16 tcgen05 kernels, fp32 accumulation)
    space_filling_curves_ext     :=  fastpcc_b200.space_filling_curves_ext
    rans_ext_cpp                 :=  the reference's own compiled coders (oracle/_ref)

at the baseline_r1 topology (BASELINE configs[3]) with seeded parameters.  Checked: the bitstream decodes (encoder and
decoder rebuild identical float features, or the range decoder desynchronises); the stride-2 geometry -- the part the
entropy model codes LOSSLESSLY -- comes back exactly; the decoder returns exactly the signalled number of points; rate
and D1 PSNR agree with the fp32 run of the same model code on the oracle's CPU MinkowskiEngine stand-in
(tests/golden/lossy_v2_golden.json) within the tolerances written below."""
import json
import os.path as osp
import zipfile

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = osp.dirname(osp.dirname(osp.abspath(__file__)))
PYREF = osp.join(ROOT, 'oracle', '_ref', 'pyref.zip')

BPP_ABS_TOL = 5e-3      # bits per point; measured on B200: identical byte counts (30.2752 / 39.8107 bpp on both backends)
TIE_SLACK = 8           # points lost to exact ties at the top-k threshold (of 6 000 - 20 000)
PSNR_ABS_TOL = 1e-2     # dB; measured: 63.284 vs 63.283 and 63.177 vs 63.177 (BASELINE north star: equal to 3 decimals)


@pytest.fixture(scope='module')
def ref_lossy(tmp_path_factory):
    from oracle import build_ref
    if build_ref.REF_ROOT and osp.isdir(osp.join(build_ref.REF_ROOT, 'models')):
        ref_root = build_ref.REF_ROOT
    elif osp.isfile(PYREF):
        ref_root = str(tmp_path_factory.mktemp('pyref'))
        with zipfile.ZipFile(PYREF) as z:
            z.extractall(ref_root)
    else:
        pytest.skip('reference Python not staged (set FASTPCC_REFERENCE_ROOT to a checkout of the reference, or run oracle/build_ref.py there)')
    from tests import ref_import
    from fastpcc_b200 import me, space_filling_curves_ext
    rans = build_ref.load_ref('rans_ext_cpp')
    if rans is None:
        pytest.skip('oracle/_ref/rans_ext_cpp not built')
    yield ref_import.import_reference_lossy_v2(ref_root, me, rans=rans, morton_ext=space_filling_curves_ext)
    # the reference model switches MinkowskiEngine's process-wide state (lossy_coord_v2/model.py:35,127-135): restore it
    me.set_sparse_tensor_operation_mode(me.SparseTensorOperationMode.SEPARATE_COORDINATE_MANAGER)
    me.clear_global_coordinate_manager()


def _cases():
    from tests.golden.lossy_cases import CASES
    gold = {g['name']: g for g in json.load(open(osp.join(ROOT, 'tests', 'golden', 'lossy_v2_golden.json')))['cases']}
    return [(c, gold[c['name']]) for c in CASES]


@pytest.mark.parametrize('case,gold', _cases(), ids=[c['name'] for c, _ in _cases()])
def test_unmodified_reference_lossy_v2_on_the_me_shim(ref_lossy, case, gold):
    from fastpcc_b200 import metrics
    from tests.golden.make_lossy_golden import run_case, stride2_sha
    xyz, data, rec = run_case(ref_lossy, case, device='cuda')
    # top-k pruning keeps scores strictly above the k-th value (lossy_coord_v2/layers.py:166-176): candidates that tie
    # with it are dropped, in the reference as here; fp16 features make such ties slightly more frequent than fp32
    assert xyz.shape[0] - TIE_SLACK <= rec.shape[0] <= xyz.shape[0] == gold['n_rec']
    assert stride2_sha(rec, xyz.min(0))[0] == gold['stride2_sha256']          # lossless part: exact
    bpp = len(data) * 8 / xyz.shape[0]
    err = metrics.pc_error(torch.from_numpy(xyz).cuda(), torch.from_numpy(np.ascontiguousarray(rec)).int().cuda(), 2 ** case['bits'])
    psnr = err['mseF,PSNR (p2point)']
    print(f"{case['name']}: bpp {bpp:.4f} (fp32 oracle {gold['bpp']:.4f}), D1 PSNR {psnr:.3f} dB (fp32 oracle {gold['d1_psnr']:.3f})")
    assert abs(bpp - gold['bpp']) <= BPP_ABS_TOL
    assert abs(psnr - gold['d1_psnr']) <= PSNR_ABS_TOL
    # a second encode gives the same bytes (fixed accumulation order: no atomics on the float path)
    _, data2, _ = run_case(ref_lossy, case, device='cuda')
    assert data2 == data
