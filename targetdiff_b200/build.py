"""Build libtdiff.so in-tree with nvcc for sm_100a (no torch involvement: the library only links cudart).

    python -m targetdiff_b200.build [--force] [--verbose]

Outputs `targetdiff_b200/libtdiff.so` (git-ignored, but it travels to the GPU box with the gpurun snapshot).
"""
import concurrent.futures
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
# TDIFF_VARIANT=<name> (developer switch, with TDIFF_NVCC_EXTRA): objects in csrc/build_<name>, library libtdiff_<name>.so -- load it with
# TDIFF_LIB=... for an A/B of two kernel builds in one GPU call
_VARIANT = os.environ.get('TDIFF_VARIANT', '')
OBJ = os.path.join(CSRC, 'build' + ('_' + _VARIANT if _VARIANT else ''))
LIB = os.path.join(HERE, 'libtdiff%s.so' % ('_' + _VARIANT if _VARIANT else ''))
SOURCES = ['engine.cu', 'knn.cu', 'edge_const.cu', 'node_ops.cu', 'edge_mlp.cu', 'edge_mlp_tc.cu', 'edge_mlp_v4.cu', 'aggregate.cu', 'sampler.cu', 'stability.cu', 'prop.cu']
HEADERS = ['tdiff_common.cuh', 'sampler.cuh', os.path.join('..', '..', 'include', 'tdiff.h')]
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17', '-Xcompiler', '-fPIC',
              '-Xcompiler', '-fvisibility=hidden', '-Xptxas', '-v']
# developer switch, e.g. TDIFF_NVCC_EXTRA=-DTDIFF_V3_TIMELINE (clock64 timeline stamps in edge_mlp_v3, see tools/v3_timeline.py)
NVCC_FLAGS += os.environ.get('TDIFF_NVCC_EXTRA', '').split()


def nvcc_path():
    p = shutil.which('nvcc') or '/usr/local/cuda/bin/nvcc'
    if not os.path.exists(p):
        raise RuntimeError('nvcc not found: libtdiff.so cannot be built (there is no CPU fallback)')
    return p


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    nvcc = nvcc_path()
    os.makedirs(OBJ, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS]
    jobs = []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        obj = os.path.join(OBJ, s.replace('.cu', '.o'))
        if force or _stale(obj, [src] + hdrs):
            jobs.append((src, obj))

    def compile_one(job):
        src, obj = job
        cmd = [nvcc] + NVCC_FLAGS + ['-c', src, '-o', obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        return job, r

    with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        for (src, obj), r in ex.map(compile_one, jobs):
            if verbose or r.returncode != 0:
                sys.stderr.write(r.stdout + r.stderr)
            if r.returncode != 0:
                raise RuntimeError('nvcc failed on %s' % src)
            with open(obj + '.log', 'w') as f:      # ptxas -v output (registers / spills / smem) kept beside the object
                f.write(r.stdout + r.stderr)
    objs = [os.path.join(OBJ, s.replace('.cu', '.o')) for s in SOURCES]
    if force or jobs or _stale(LIB, objs):
        cmd = [nvcc, '-shared', '-gencode', 'arch=compute_100a,code=sm_100a', '-o', LIB] + objs
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError('link failed')
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='--verbose' in sys.argv))
