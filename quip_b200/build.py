"""Build libquip_b200.so (all CUDA kernels + the C ABI) in-tree for sm_100a.

    python -m quip_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU; the .so travels to the GPU box with the snapshot.
"""
import argparse
import concurrent.futures as cf
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
OBJ = os.path.join(HERE, 'build')
LIB = os.path.join(HERE, 'libquip_b200.so')
SOURCES = ['api.cu', 'pack.cu', 'rot.cu', 'rot_small.cu', 'rot_fewtok.cu', 'rot_side.cu', 'rot_side_fewtok.cu', 'glue.cu', 'vecquant.cu', 'ldlq.cu', 'hessian.cu', 'qgemm_skinny.cu', 'qgemv.cu', 'qgemm_tc.cu', 'attn_decode.cu']
NVCC = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
         '-Xcompiler', '-fPIC', '--expt-relaxed-constexpr']


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    headers = [os.path.join(CSRC, 'common.cuh'), os.path.join(CSRC, 'tc_common.cuh'), os.path.join(os.path.dirname(HERE), 'include', 'quip_b200.h')]
    jobs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src.replace('.cu', '.o'))
        if force or _stale(o, [s] + headers):
            cmd = [NVCC] + FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-c', s, '-o', o]
            jobs.append((src, cmd))

    def run(job):
        src, cmd = job
        r = subprocess.run(cmd, capture_output=True, text=True)
        return src, r

    with cf.ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        for src, r in ex.map(run, jobs):
            if verbose or r.returncode:
                sys.stderr.write(f'--- {src}\n{r.stdout}{r.stderr}\n')
            if r.returncode:
                raise RuntimeError(f'nvcc failed on {src}')
    objs = [os.path.join(OBJ, s.replace('.cu', '.o')) for s in SOURCES]
    if force or jobs or _stale(LIB, objs):
        cmd = [NVCC, '-shared', '-o', LIB] + objs + ['-gencode', 'arch=compute_100a,code=sm_100a']
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError('link failed')
    return LIB


if __name__ == '__main__':
    ap = argparse.ArgumentParser()
    ap.add_argument('--force', action='store_true')
    ap.add_argument('--verbose', action='store_true')
    a = ap.parse_args()
    print(build(a.force, a.verbose))
