"""Builds libptb_b200.so (sm_100a only) in-tree with nvcc.  Used by __graft_entry__.build() and by hand:
    python pointtinybenchmark_b200/csrc/build.py [--force] [--verbose]
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(os.path.dirname(HERE), 'libptb_b200.so')
SOURCES = ['capi.cu', 'gather.cu', 'linear.cu', 'negmask.cu', 'refine.cu', 'gridbag.cu', 'mil.cu', 'p2p.cu', 'nms.cu', 'conv_tc.cu', 'tower_bwd.cu', 'wgrad_tc.cu', 'assign.cu', 'lsap.cu', 'rpn.cu', 'loss_bwd.cu', 'roi_align.cu']
ARCH = ['-gencode', 'arch=compute_100a,code=sm_100a']
FLAGS = ['-O3', '-std=c++17', '-lineinfo', '-Xcompiler', '-fPIC', '--expt-relaxed-constexpr', '-Xptxas', '-v']


def _nvcc():
    for c in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError('nvcc not found')


def needs_build(srcs):
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    import glob
    deps = [os.path.join(HERE, s) for s in srcs] + glob.glob(os.path.join(HERE, '*.cuh')) + [os.path.join(HERE, '..', '..', 'include', 'ptb_b200.h'), __file__]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(HERE, s))]
    if not force and not needs_build(srcs):
        return OUT
    nvcc = _nvcc()
    objdir = os.path.join(HERE, 'build')
    os.makedirs(objdir, exist_ok=True)

    def cc(src):
        obj = os.path.join(objdir, src.replace('.cu', '.o'))
        cmd = [nvcc] + ARCH + FLAGS + ['-c', os.path.join(HERE, src), '-o', obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f'nvcc failed for {src}:\n{r.stdout}\n{r.stderr}')
        return obj, r.stderr

    with ThreadPoolExecutor(max_workers=8) as ex:
        res = list(ex.map(cc, srcs))
    if verbose:
        for _, log in res:
            print(log)
    cmd = [nvcc] + ARCH + ['-shared', '-o', OUT] + [o for o, _ in res] + ['-lcudart']
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f'link failed:\n{r.stdout}\n{r.stderr}')
    return OUT


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='--verbose' in sys.argv))
