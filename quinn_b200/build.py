"""Build the CUDA library in-tree:  python -m quinn_b200.build [--force] [-v]

Translation units under quinn_b200/csrc/*.cu are compiled for sm_100a only
(-gencode arch=compute_100a,code=sm_100a -lineinfo), in parallel, and linked into
quinn_b200/lib/libquinn_b200.so (git-ignored, but it travels to the GPU box).  A stamp file next to the
library records the SHA-256 of every source; build() recompiles whenever the sources no longer match it.
"""
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, 'csrc')
UNITS = ['qb_kernels.cu', 'qb_launch.cu', 'qb_grad_tc.cu', 'qb_grad_tc128.cu', 'qb_value_tc3.cu', 'qb_post.cu']
HEADERS = ['qb_device.cuh', 'qb_chain.cuh', 'qb_stream.cuh', 'qb_hvp.cuh', 'qb_kfac.cuh', 'qb_jac.cuh', 'qb_swag.cuh', 'qb_nuts.cuh', 'qb_pt.cuh', 'qb_tcgen05.cuh', 'qb_tc.cuh', 'qb_tc3.cuh', 'qb_tcg.cuh', 'qb_tg8.cuh', 'qb_tg8_plan.h', 'qb_grad_tc.h', 'qb_grad_tc128.h', 'qb_value_tc3.h', 'qb_plan.h', 'qb_launch.h']
DEPS = [os.path.join(CSRC, f) for f in UNITS + HEADERS] + [os.path.join(ROOT, 'include', 'quinn_b200.h')]
OUT = os.path.join(HERE, 'lib', 'libquinn_b200.so')
STAMP = OUT + '.srchash'
OBJDIR = os.path.join(ROOT, 'build', 'obj')


def source_hash():
    h = hashlib.sha256()
    for d in DEPS:
        h.update(os.path.basename(d).encode())
        with open(d, 'rb') as f:
            h.update(f.read())
    return h.hexdigest()


def needs_build():
    if not os.path.exists(OUT) or not os.path.exists(STAMP):
        return True
    with open(STAMP) as f:
        return f.read().strip() != source_hash()


def _nvcc():
    return os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')


def _unit_deps(unit):
    """The unit and every header it includes (transitively) from csrc/ or include/."""
    import re
    seen, todo = [], [os.path.join(CSRC, unit)]
    while todo:
        f = todo.pop()
        if f in seen or not os.path.exists(f):
            continue
        seen.append(f)
        with open(f) as fh:
            for inc in re.findall(r'#include\s+"([^"]+)"', fh.read()):
                for d in (CSRC, os.path.join(ROOT, 'include')):
                    if os.path.exists(os.path.join(d, inc)):
                        todo.append(os.path.join(d, inc))
    return sorted(seen)


def _unit_hash(unit):
    h = hashlib.sha256()
    for d in _unit_deps(unit):
        h.update(os.path.basename(d).encode())
        with open(d, 'rb') as f:
            h.update(f.read())
    return h.hexdigest()


def _compile(unit, verbose, force=False):
    obj = os.path.join(OBJDIR, unit.replace('.cu', '.o'))
    stamp, uh = obj + '.srchash', _unit_hash(unit)
    if not force and os.path.exists(obj) and os.path.exists(stamp) and open(stamp).read().strip() == uh:
        return unit, obj, subprocess.CompletedProcess([], 0, '', '')        # object is current (only its own sources count)
    cmd = [_nvcc(), '-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17', '-c',
           '-Xcompiler', '-fPIC', '-I', os.path.join(ROOT, 'include'), '-I', CSRC, '-o', obj, os.path.join(CSRC, unit)]
    if verbose:
        cmd[1:1] = ['-Xptxas', '-v']
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode == 0:
        with open(stamp, 'w') as f:
            f.write(uh + '\n')
    return unit, obj, res


def build(force=False, verbose=False):
    if not force and not needs_build():
        return OUT
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    os.makedirs(OBJDIR, exist_ok=True)
    with ThreadPoolExecutor(len(UNITS)) as ex:
        results = list(ex.map(lambda u: _compile(u, verbose, force), UNITS))
    objs = []
    for unit, obj, res in results:
        if res.returncode != 0:
            sys.stderr.write(res.stdout + res.stderr)
            raise RuntimeError(f'nvcc failed compiling {unit}')
        if verbose:
            sys.stderr.write(res.stderr)
        objs.append(obj)
    res = subprocess.run([_nvcc(), '-gencode', 'arch=compute_100a,code=sm_100a', '--shared', '-o', OUT] + objs,
                         capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError('nvcc failed linking libquinn_b200.so')
    with open(STAMP, 'w') as f:
        f.write(source_hash() + '\n')
    return OUT


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
