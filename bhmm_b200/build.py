"""Build libbhmm_b200.so (hand-written sm_100a CUDA kernels + C ABI) in-tree with nvcc.

    python bhmm_b200/build.py            # incremental
    python bhmm_b200/build.py --force

The shared library lands next to this file (bhmm_b200/libbhmm_b200.so) so that it travels with the source
tree; it is git-ignored.  nvcc cross-compiles for sm_100a without a GPU.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
OBJ = os.path.join(CSRC, '_obj')
LIB = os.path.join(HERE, 'libbhmm_b200.so')
SOURCES = ['lane_inst_a.cu', 'lane_inst_b.cu', 'lane_inst_c.cu', 'lane_inst_d.cu', 'lane_inst_e.cu', 'lane_inst_f.cu',
           'lane_dispatch.cu', 'team_kernels.cu', 'panel_kernels.cu', 'lane_viterbi.cu', 'scan_kernels.cu', 'frame_kernels.cu', 'tmatrix_kernels.cu', 'init_kernels.cu', 'certify.cu', 'sample_kernels.cu', 'capi.cu', 'engine.cu', 'transfer.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '--expt-relaxed-constexpr', '-Xcompiler', '-fPIC', '-Xptxas', '-v']


def _nvcc():
    for cand in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    raise RuntimeError('nvcc not found')


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, defines=(), libname=None):
    """Compile and link.  `defines` (e.g. ['-DLANE_MINB_F=6']) and `libname` build a tuning variant next to the
    default library (its objects go to a separate directory)."""
    global OBJ, LIB
    if libname:
        OBJ = os.path.join(CSRC, '_obj_' + libname)
        LIB = os.path.join(HERE, 'lib%s.so' % libname)
    os.makedirs(OBJ, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.h', '.cuh'))]
    headers.append(os.path.join(os.path.dirname(HERE), 'include', 'bhmm_b200.h'))
    nvcc = _nvcc()
    jobs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src.replace('.cu', '.o'))
        if force or _stale(o, [s] + headers):
            jobs.append((s, o))

    def compile_one(job):
        s, o = job
        cmd = [nvcc] + NVCC_FLAGS + list(defines) + ['-c', s, '-o', o]
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        with open(o + '.log', 'w') as fh:
            fh.write(' '.join(cmd) + '\n' + r.stdout)
        if r.returncode != 0:
            raise RuntimeError('nvcc failed for %s:\n%s' % (s, r.stdout))
        if verbose:
            print(r.stdout)
        return o

    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        list(ex.map(compile_one, jobs))
    objs = [os.path.join(OBJ, s.replace('.cu', '.o')) for s in SOURCES]
    if force or jobs or _stale(LIB, objs):
        cmd = [nvcc, '-shared', '-o', LIB] + objs + ['-gencode', 'arch=compute_100a,code=sm_100a']
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if r.returncode != 0:
            raise RuntimeError('link failed:\n' + r.stdout)
    return LIB


if __name__ == '__main__':
    # -DNAME=VALUE defines and --nvcc=<flag> extra compiler flags (e.g. --nvcc=-Xptxas --nvcc=-O2) for variant builds
    defs = [a for a in sys.argv[1:] if a.startswith('-D')] + [a.split('=', 1)[1] for a in sys.argv[1:] if a.startswith('--nvcc=')]
    name = None
    for a in sys.argv[1:]:
        if a.startswith('--name='):
            name = a.split('=', 1)[1]
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv, defines=defs, libname=name))
