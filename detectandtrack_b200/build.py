"""In-tree build of libdt_b200.so (sm_100a only) and of the oracle's helpers.

    python -m detectandtrack_b200.build [--force]

nvcc cross-compiles without a GPU.  Objects/outputs are git-ignored but travel
to the GPU box with the gpurun snapshot.
"""
import os, subprocess, sys, shutil
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, 'csrc')
OBJ = os.path.join(HERE, 'build')
LIBDIR = os.path.join(HERE, 'lib')
LIB = os.path.join(LIBDIR, 'libdt_b200.so')

NVCC = os.environ.get('NVCC', shutil.which('nvcc') or '/usr/local/cuda/bin/nvcc')
ARCH = ['-gencode', 'arch=compute_100a,code=sm_100a']
COMMON = ['-O3', '-std=c++17', '-lineinfo', '-Xcompiler', '-fPIC', '--expt-relaxed-constexpr',
          '-I' + os.path.join(ROOT, 'include')]
# bit-exact integer/index kernels: no FMA contraction anywhere in these units
EXACT = {'boxes.cu', 'lsa.cu', 'proposals.cu', 'detections.cu', 'targets.cu'}


def _newer(src, dst, extra=()):
    if not os.path.exists(dst):
        return True
    t = os.path.getmtime(dst)
    return any(os.path.getmtime(s) > t for s in (src,) + tuple(extra))


def build_lib(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    os.makedirs(LIBDIR, exist_ok=True)
    headers = tuple(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.cuh', '.h')))
    headers += tuple(os.path.join(ROOT, 'include', f) for f in os.listdir(os.path.join(ROOT, 'include')) if f.endswith('.h'))
    srcs = sorted(f for f in os.listdir(CSRC) if f.endswith('.cu'))
    jobs = []
    objs = []
    for f in srcs:
        src = os.path.join(CSRC, f)
        obj = os.path.join(OBJ, f[:-3] + '.o')
        objs.append(obj)
        if force or _newer(src, obj, headers):
            cmd = [NVCC] + ARCH + COMMON + (['-fmad=false'] if f in EXACT else []) + \
                  (['-Xptxas', '-v'] if verbose else []) + ['-c', src, '-o', obj]
            jobs.append(cmd)

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError('nvcc failed: %s\n%s\n%s' % (' '.join(cmd), r.stdout, r.stderr))
        if verbose:
            print(r.stderr)
    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        list(ex.map(run, jobs))
    if jobs or force or not os.path.exists(LIB):
        cmd = [NVCC] + ARCH + ['-shared', '-Xcompiler', '-fPIC', '-o', LIB] + objs + ['-lcudart_static', '-ldl', '-lpthread', '-lrt']     # nvJPEG is dlopen'ed by jpeg.cu, not linked
        run(cmd)
    return LIB


if __name__ == '__main__':
    print(build_lib(force='--force' in sys.argv, verbose='-v' in sys.argv))
