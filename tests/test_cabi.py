"""The C-ABI library builds, loads and exports every symbol include/qcmrf_b200.h
declares; without a GPU the product fails loudly (no CPU fallback).  CPU only, no
compute calls."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT, has_cuda
from qcmrf_b200 import _native, fusion


def _header_functions():
    src = open(os.path.join(ROOT, 'include', 'qcmrf_b200.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(qcm_[a-z_0-9]+)\s*\(', src)))


def test_library_exports_every_declared_symbol(native_built):
    declared = _header_functions()
    assert sorted(_native.SYMBOLS) == declared
    lib = ctypes.CDLL(native_built)
    for name in declared:
        assert hasattr(lib, name), name
    out = subprocess.run(['nm', '-D', '--defined-only', native_built], capture_output=True, text=True).stdout
    exported = sorted(l.split()[-1] for l in out.splitlines() if ' T ' in l)
    assert exported == declared            # nothing else leaks out of the library
    assert lib.qcm_abi_version() == 1
    assert lib.qcm_small_max_qubits(32) == 13 and lib.qcm_small_max_qubits(64) == 13


def test_op_struct_layout_matches_header(native_built, tmp_path):
    """qcm_op as numpy sees it == as the C compiler lays it out."""
    src = r'''
    #include <stdio.h>
    #include <stddef.h>
    #include "qcmrf_b200.h"
    int main(void){ printf("%zu %zu %zu %zu %zu %zu", sizeof(qcm_op), offsetof(qcm_op, n_active_in),
        offsetof(qcm_op, ctrl), offsetof(qcm_op, table_off), sizeof(qcm_timing), offsetof(qcm_op, flags)); return 0; }
    '''
    exe = str(tmp_path / 'qcm_layout_test')
    subprocess.run(['gcc', '-x', 'c', '-', '-I', os.path.join(ROOT, 'include'), '-o', exe], input=src, text=True, check=True)
    vals = list(map(int, subprocess.run([exe], capture_output=True, text=True).stdout.split()))
    d = fusion.OP_DTYPE
    assert vals[0] == d.itemsize
    assert vals[1] == d.fields['n_active_in'][1] and vals[2] == d.fields['ctrl'][1]
    assert vals[3] == d.fields['table_off'][1] and vals[5] == d.fields['flags'][1]
    assert vals[4] == ctypes.sizeof(_native.QcmTiming)


@pytest.mark.skipif(has_cuda(), reason='this checks the GPU-less failure mode')
def test_fails_loudly_without_a_gpu(native_built):
    lib = _native.lib()
    h = ctypes.c_void_p()
    rc = lib.qcm_create(ctypes.byref(h), 0, 10, 64, None, None)
    assert rc == -5 and not h.value                       # QCM_ERR_NO_DEVICE
    assert b'no CUDA device' in lib.qcm_last_error(None)
    with pytest.raises(_native.NativeError):
        _native.Handle(10, 'double')
    from qcmrf_b200 import QCMRF, B200Simulator
    with pytest.raises(_native.NativeError):
        B200Simulator().run(QCMRF([[0, 1]], [-0.1] * 4), shots=10)
    with pytest.raises(_native.NativeError):
        B200Simulator(small_batch=False).run(QCMRF([[0, 1]], [-0.1] * 4), shots=10)


def test_null_and_bad_arguments_return_codes(native_built):
    lib = _native.lib()
    assert lib.qcm_device_count(None) == -1
    assert lib.qcm_create(None, 0, 4, 32, None, None) == -1
    h = ctypes.c_void_p()
    assert lib.qcm_create(ctypes.byref(h), 0, 4, 16, None, None) == -1      # bad precision
    assert lib.qcm_create(ctypes.byref(h), 0, 99, 32, None, None) == -1     # absurd width
    assert lib.qcm_run_program(None, None, 0, None, 0) == -1
    assert lib.qcm_destroy(None) == 0
    k = ctypes.c_double()
    assert lib.qcm_run_batch_small(0, 32, 0, None, None, None, None, 0, None, None, None, None, None, None,
                                   0, 0, None, None, None, ctypes.byref(k)) == -1
