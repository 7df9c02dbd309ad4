"""In-tree nvcc build of libfastpcc_b200.so (sm_100a only; no JIT cache, the .so travels with the repo)."""
import os
import os.path as osp
import subprocess
import sys

HERE = osp.dirname(osp.abspath(__file__))
CSRC = osp.join(HERE, 'csrc')
OUT_DIR = osp.join(HERE, '_C')
SO = osp.join(OUT_DIR, 'libfastpcc_b200.so')
SOURCES = ['common.cu', 'coords.cu', 'igemm_simt.cu', 'igemm_tc.cu', 'ops_api.cu', 'entropy.cu', 'rans.cu', 'frontend.cu', 'container.cu', 'metrics.cu', 'train.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC', '--expt-relaxed-constexpr']


def _newest_src():
    t = 0.0
    for root, _, files in os.walk(CSRC):
        for f in files:
            t = max(t, osp.getmtime(osp.join(root, f)))
    t = max(t, osp.getmtime(osp.join(HERE, '..', 'include', 'fastpcc_b200.h')))
    return t


def _compile_and_link(out_dir, extra_flags=(), verbose=False):
    """Compiles every source in parallel into out_dir/obj, writes out_dir/ptxas.log and links out_dir/libfastpcc_b200.so."""
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    os.makedirs(osp.join(out_dir, 'obj'), exist_ok=True)
    procs, objs = [], []
    for src in SOURCES:
        obj = osp.join(out_dir, 'obj', src.replace('.cu', '.o'))
        objs.append(obj)
        cmd = [nvcc] + NVCC_FLAGS + list(extra_flags) + ['-Xptxas', '-v', '-c', osp.join(CSRC, src), '-o', obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    for src, p in procs:
        out, _ = p.communicate()
        log.append(f'==== {src}\n{out}')
        if p.returncode != 0:
            sys.stderr.write(out)
            raise RuntimeError(f'nvcc failed on {src}')
    with open(osp.join(out_dir, 'ptxas.log'), 'w') as f:
        f.write('\n'.join(log))
    if verbose:
        print('\n'.join(log))
    so = osp.join(out_dir, 'libfastpcc_b200.so')
    subprocess.run([nvcc, '-shared', '-o', so] + objs, check=True)
    return so


def build(force=False, verbose=False):
    if not force and osp.isfile(SO) and osp.getmtime(SO) >= _newest_src():
        return SO
    return _compile_and_link(OUT_DIR, verbose=verbose)


def build_variant(name, extra_flags):
    """Diagnostic builds for A/B runs in ONE GPU call: the same sources with extra nvcc flags (e.g. ['-DFPCC_TC_TRACE'])
    into _C/variants/<name>/libfastpcc_b200.so, selected at run time with FPCC_LIB_PATH (fastpcc_b200/_lib.py).  The
    default library is untouched."""
    return _compile_and_link(osp.join(OUT_DIR, 'variants', name), extra_flags)


if __name__ == '__main__':
    print(build(force='-f' in sys.argv, verbose='-v' in sys.argv))
