"""Builds libphoenix_b200.so in-tree with nvcc for sm_100a (no JIT cache, no torch extension
machinery: the library is a plain C-ABI shared object loaded with ctypes)."""
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'libphoenix_b200.so')

ARCH = ['-gencode', 'arch=compute_100a,code=sm_100a']
COMMON = ['-std=c++17', '-O3', '-lineinfo', '--expt-relaxed-constexpr', '-Xcompiler', '-fPIC']
# translation unit -> extra flags.  The float64 kernels are the parity instantiation: no FMA
# contraction, so that products and sums round like the reference's numpy expressions.  The
# float32 kernels are the throughput instantiation: MUFU approximations for sin/cos/sqrt/div.
UNITS = {
    'pdx_tu_f32_simple.cu': ['-use_fast_math'],
    'pdx_tu_f32_bullet.cu': ['-use_fast_math'],
    'pdx_tu_f64_simple.cu': ['-fmad=false'],
    'pdx_tu_f64_bullet.cu': ['-fmad=false'],
    'pdx_tu_f32_simple_pid.cu': ['-use_fast_math'],
    'pdx_tu_f32_bullet_pid.cu': ['-use_fast_math'],
    'pdx_tu_f64_simple_pid.cu': ['-fmad=false'],
    'pdx_tu_f64_bullet_pid.cu': ['-fmad=false'],
    'pdx_abi.cu': [],
    'pdx_rollout.cu': [],
    'pdx_policy_tc.cu': [],
    'pdx_collect.cu': ['-use_fast_math'],
    'pdx_evaluate.cu': ['-use_fast_math'],
}


def _nvcc():
    for cand in (os.environ.get('NVCC'), shutil.which('nvcc'), '/usr/local/cuda/bin/nvcc'):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError('nvcc not found: libphoenix_b200.so cannot be built')


def _stale(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def build(force=False, verbose=False):
    nvcc = _nvcc()
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.cuh', '.h'))]
    headers.append(os.path.join(os.path.dirname(HERE), 'include', 'phoenix_b200.h'))
    headers.append(os.path.abspath(__file__))
    obj_dir = os.path.join(HERE, 'build')
    os.makedirs(obj_dir, exist_ok=True)
    jobs = []
    for unit, extra in UNITS.items():
        src = os.path.join(CSRC, unit)
        obj = os.path.join(obj_dir, unit.replace('.cu', '.o'))
        if force or _stale(obj, [src] + headers):
            jobs.append([nvcc] + ARCH + COMMON + extra + (['-Xptxas', '-v'] if verbose else []) + ['-c', src, '-o', obj])

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError('nvcc failed:\n' + ' '.join(cmd) + '\n' + r.stdout + r.stderr)
        return r.stderr

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        logs = list(ex.map(run, jobs))
    objs = [os.path.join(obj_dir, u.replace('.cu', '.o')) for u in UNITS]
    if force or jobs or _stale(LIB, objs):
        run([nvcc] + ARCH + ['-shared', '-o', LIB] + objs)
    if verbose:
        print('\n'.join(logs))
    return LIB


def build_timing():
    """libphoenix_b200_timing.so: the same library with -DPDX_TC_TIMING (k_policy_tc records clock64
    stamps per phase; read with pdx_policy_tc_timing, see tools/policy_tc_timing.py)."""
    build()
    nvcc = _nvcc()
    obj_dir = os.path.join(HERE, 'build')
    tobj = os.path.join(obj_dir, 'pdx_policy_tc_timing.o')
    subprocess.run([nvcc] + ARCH + COMMON + ['-DPDX_TC_TIMING', '-c', os.path.join(CSRC, 'pdx_policy_tc.cu'), '-o', tobj], check=True)
    objs = [os.path.join(obj_dir, u.replace('.cu', '.o')) for u in UNITS if u != 'pdx_policy_tc.cu'] + [tobj]
    out = os.path.join(HERE, 'libphoenix_b200_timing.so')
    subprocess.run([nvcc] + ARCH + ['-shared', '-o', out] + objs, check=True)
    return out


if __name__ == '__main__':
    if '--timing' in sys.argv:
        print(build_timing())
    else:
        print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
