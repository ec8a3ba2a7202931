"""In-tree build of the CUDA engine: nvcc -> qcmrf_b200/libqcmrf_b200.so (sm_100a only).

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'libqcmrf_b200.so')
SOURCES = ['qcm_api.cu', 'qcm_small.cu', 'qcm_mrf.cu', 'qcm_noise.cu']
HEADERS = [os.path.join(CSRC, 'qcm_kernels.cuh'), os.path.join(CSRC, 'qcm_noise.h'), os.path.join(ROOT, 'include', 'qcmrf_b200.h')]

NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC',
              '-Xcompiler', '-fvisibility=hidden', '-Xcompiler', '-O3']


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + HEADERS
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


HOST_LIB = os.path.join(HERE, '_qcm_host.so')
HOST_SRC = os.path.join(CSRC, 'qcm_host.c')


def build_host(force=False, verbose=False):
    """gcc -> qcmrf_b200/_qcm_host.so: result formatting through the CPython C API (no CUDA)."""
    if not force and os.path.exists(HOST_LIB) and os.path.getmtime(HOST_LIB) >= os.path.getmtime(HOST_SRC):
        return HOST_LIB
    import sysconfig
    cc = shutil.which('gcc') or shutil.which('cc')
    if cc is None:
        raise RuntimeError('gcc not found: cannot build qcmrf_b200/_qcm_host.so')
    cmd = [cc, '-O2', '-ffp-contract=off', '-shared', '-fPIC', '-I', sysconfig.get_paths()['include'], HOST_SRC, '-o', HOST_LIB, '-lm']
    if verbose:
        print(' '.join(cmd))
    subprocess.check_call(cmd)
    return HOST_LIB


def build_native(force=False, verbose=False):
    """Compile the engine if sources are newer than the library. Returns the .so path."""
    build_host(force, verbose)
    if not force and not _stale():
        return LIB
    nvcc = shutil.which('nvcc') or '/usr/local/cuda/bin/nvcc'
    if not os.path.exists(nvcc):
        raise RuntimeError('nvcc not found: cannot build qcmrf_b200 CUDA engine')
    objs = []
    bdir = os.path.join(HERE, 'build')
    os.makedirs(bdir, exist_ok=True)
    procs = []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        if not os.path.exists(src):
            continue
        obj = os.path.join(bdir, s.replace('.cu', '.o'))
        cmd = [nvcc] + NVCC_FLAGS + ['-I', os.path.join(ROOT, 'include'), '-I', CSRC, '-c', src, '-o', obj]
        if verbose:
            print(' '.join(cmd))
        procs.append((subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT), cmd))
        objs.append(obj)
    for p, cmd in procs:
        out, _ = p.communicate()
        if p.returncode:
            raise RuntimeError('nvcc failed:\n' + ' '.join(cmd) + '\n' + out.decode())
    cmd = [nvcc, '-shared', '-o', LIB] + objs + ['-gencode', 'arch=compute_100a,code=sm_100a', '-cudart', 'static']
    subprocess.check_call(cmd)
    return LIB


if __name__ == '__main__':
    print(build_native(force='--force' in sys.argv, verbose=True))
