"""Compile the CUDA sources in csrc/ for sm_100a into libdsdf_b200.so (in-tree, next to this file).

    python -m diffsdfsim_b200.build [--force]

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box with the snapshot.
"""
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
OUT = os.path.join(HERE, 'libdsdf_b200.so')
OBJ = os.path.join(HERE, 'csrc', '_build')
NVCC = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
         '-Xcompiler', '-fPIC', '-Xptxas', '-v', '--expt-relaxed-constexpr'] + os.environ.get('DSDF_EXTRA_FLAGS', '').split()
# Per-file extras.  The contact refinement makes round-off-level decisions (arg-min ties in Frank-Wolfe, which
# body's normal to use on flat-flat contacts) that the reference takes with un-fused IEEE multiply/add (torch
# element-wise ops): compile that file without FMA contraction so the same ties break the same way.
_NOFMA = ['-fmad=false']
_PHASES = ['-DDSDF_PHASE_PROFILE'] if os.environ.get('DSDF_PHASE_PROFILE') else []
EXTRA = {'dsdf_contacts_bwd.cu': _NOFMA, 'dsdf_contacts.cu': _NOFMA + _PHASES
         + (['-DDSDF_CONTACT_MINBLOCKS=' + os.environ['DSDF_CONTACT_MINBLOCKS']] if os.environ.get('DSDF_CONTACT_MINBLOCKS') else []),
         'dsdf_dynsolve.cu': _PHASES}


def _sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith('.cu'))


def _stamp():
    h = hashlib.sha1()
    for root in (CSRC, os.path.join(os.path.dirname(HERE), 'include')):
        for f in sorted(os.listdir(root)):
            if f.endswith(('.cu', '.cuh', '.h')):
                with open(os.path.join(root, f), 'rb') as fh:
                    h.update(f.encode() + fh.read())
    h.update((' '.join(FLAGS) + repr(sorted(EXTRA.items()))).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    stamp_file = os.path.join(OBJ, 'stamp')
    stamp = _stamp()
    if not force and os.path.exists(OUT) and os.path.exists(stamp_file) and open(stamp_file).read() == stamp:
        return OUT
    srcs = _sources()

    def cc(src):
        obj = os.path.join(OBJ, os.path.basename(src)[:-3] + '.o')
        r = subprocess.run([NVCC] + FLAGS + EXTRA.get(os.path.basename(src), []) + ['-c', src, '-o', obj],
                           capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError('nvcc failed for %s:\n%s' % (src, r.stderr))
        with open(obj + '.ptxas.log', 'w') as fh:
            fh.write(r.stderr)
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=8) as ex:
        objs = list(ex.map(cc, srcs))
    r = subprocess.run([NVCC, '-shared', '-o', OUT] + objs + ['-gencode', 'arch=compute_100a,code=sm_100a'],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError('link failed:\n' + r.stderr)
    with open(stamp_file, 'w') as fh:
        fh.write(stamp)
    return OUT


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose=True))
