"""The drop-in boundary on the GPU: the reference's OWN, UNMODIFIED `models/convolutional/lossl_coord_int/model.py`
and `lib/int_sparse_conv/cuda_ops.py` (Python loop over kernel offsets, pair-list kernel maps, per-layer requant
calls, CPU range coder -- everything as the reference wrote it) run on this repository's extension shim:

    lib.int_sparse_conv.build.int_sparse_conv_ext  :=  fastpcc_b200.int_sparse_conv.ext      (binding.cu:114-145)
    space_filling_curves_ext                       :=  fastpcc_b200.space_filling_curves_ext (morton3d.cu:39-76)
    torchsparse.SparseTensor                       :=  fastpcc_b200.sparse_tensor.SparseTensor
    simple_rans_ext_cpp                            :=  the reference's own C++ coder compiled into oracle/_ref

and must reproduce tests/golden/int_codec_golden.json (minted by the same Python on CPU stand-ins of the extension)
byte for byte.  The reference tree is not present on the GPU box: oracle/build_ref.py stages its .py files into the
git-ignored oracle/_ref/pyref.zip (it travels with the snapshot), extracted here into a temporary directory.
"""
import hashlib
import json
import os.path as osp
import zipfile

import numpy as np
import pytest
import torch

from fastpcc_b200 import synth

pytestmark = pytest.mark.gpu

ROOT = osp.dirname(osp.dirname(osp.abspath(__file__)))
PYREF = osp.join(ROOT, 'oracle', '_ref', 'pyref.zip')


@pytest.fixture(scope='module')
def ref_model_module(tmp_path_factory):
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
    from fastpcc_b200 import space_filling_curves_ext
    from fastpcc_b200.int_sparse_conv import ext
    from fastpcc_b200.sparse_tensor import SparseTensor
    simple_rans = build_ref.load_ref('simple_rans_ext_cpp')
    if simple_rans is None:
        pytest.skip('oracle/_ref/simple_rans_ext_cpp not built')
    return ref_import.import_reference_model(ref_root, ext, sparse_tensor_cls=SparseTensor, morton_ext=space_filling_curves_ext,
                                             simple_rans=simple_rans, rans=build_ref.load_ref('rans_ext_cpp'))


def _cases():
    from tests.golden.int_codec_cases import CASES
    gold = json.load(open(osp.join(ROOT, 'tests', 'golden', 'int_codec_golden.json')))['cases']
    return list(zip(CASES, gold))


@pytest.mark.parametrize('case,gold', _cases(), ids=[c['name'] for c, _ in _cases()])
def test_unmodified_reference_model_on_the_extension_shim(ref_model_module, case, gold):
    from tests import ref_import
    from tests.golden.int_codec_cases import case_cloud
    cfg = case['cfg']
    sd = synth.make_lossl_int_state_dict(seed=7, **{k: v for k, v in cfg.items() if k != 'skip_top_scales_num'})
    m = ref_import.build_reference_model(ref_model_module, cfg, sd, device='cuda')
    xyz = torch.from_numpy(synth.with_batch(case_cloud(case))).cuda()
    with torch.no_grad():
        data = m.compress(xyz)
        assert len(data) == gold['n_bytes']
        assert hashlib.sha256(data).hexdigest() == gold['bitstream_sha256']
        rec = m.decompress(data).cpu().numpy()
    assert hashlib.sha256(np.ascontiguousarray(rec.astype('<i4')).tobytes()).hexdigest() == gold['decoded_sha256']
    # and the B200-native twin of the same model gives the same bytes (both sides of the boundary agree)
    from fastpcc_b200.lossl_coord_int import Config, Model
    twin = Model(Config(**cfg), device='cuda').load_numpy_state_dict(sd).cuda()
    assert twin.compress(xyz) == data
