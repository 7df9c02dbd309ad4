import sys, os.path as osp, zipfile, tempfile
ROOT = osp.dirname(osp.dirname(osp.abspath(__file__))); sys.path.insert(0, ROOT)
import numpy as np, torch
from oracle import build_ref
from tests import ref_import
from fastpcc_b200 import me, space_filling_curves_ext, synth
from tests.golden.lossy_cases import CASES, case_cloud
from tests.golden.make_lossy_golden import run_case
ref_root = build_ref.REF_ROOT
if not ref_root or not osp.isdir(ref_root + '/models'):
    ref_root = tempfile.mkdtemp(); zipfile.ZipFile(osp.join(ROOT, 'oracle/_ref/pyref.zip')).extractall(ref_root)
ref = ref_import.import_reference_lossy_v2(ref_root, me, rans=build_ref.load_ref('rans_ext_cpp'), morton_ext=space_filling_curves_ext)
case = CASES[0]
xyz, data, rec = run_case(ref, case, device='cuda')
print(rec.dtype, rec.shape, rec.min(0), rec.max(0), xyz.min(0), xyz.max(0))
a = np.unique(rec // 2, axis=0); b = np.unique(xyz // 2, axis=0)
sa = set(map(tuple, a.tolist())); sb = set(map(tuple, b.tolist()))
print(len(sa), len(sb), len(sa & sb), list(sa - sb)[:5], list(sb - sa)[:5])
off = xyz.min(0)
a = np.unique((rec - off) // 2, axis=0); b = np.unique((xyz - off) // 2, axis=0)
sa = set(map(tuple, a.tolist())); sb = set(map(tuple, b.tolist()))
print('rel to min:', len(sa), len(sb), len(sa & sb))
