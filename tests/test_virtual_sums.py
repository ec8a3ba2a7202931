"""The checkpoint sums of the virtual last pass (k_expand_low_sums) against those of the materialising pass
(k_expand_low + k_group_sum), bit for bit, through the read-only tree accessor (qcm_tree_level).

A one-ulp change in one level-0 entry drops out of the tree total and almost never moves a sampled key, so the keys
cannot show it: every level of the tree is read back and compared with np.array_equal.  The finer level (-1) is stored
by the materialising pass and computed from the retained input, with the sampler's arithmetic, for the unwritten one.  Child processes run under
QCM_VIRTUAL_LAST=0 (written) and =1 (unwritten) for every QCM_LOW_SHAPE, in both precisions, at n_in = 10 (one chunk)
to 25, plus a q33 circuit through the public simulator.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
if __name__ == '__main__':                                   # child process
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.dirname(HERE))

from qcmrf_b200 import _native                              # noqa: E402
from test_engine_paths import Prog, _has_cuda               # noqa: E402

SHAPES = ('8x8', '8x10', '4x7', '2x6', '1x5')
N_INS = (10, 11, 13, 17, 21, 25)

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not _has_cuda(), reason='needs a CUDA device')]


class _Dev:
    """A device array the engine owns, for torch.as_tensor (only copied out, never written)."""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {'shape': (n,), 'typestr': '<f8', 'data': (ptr, False), 'version': 3}


def _levels(h):
    import torch
    torch.cuda.synchronize()
    out = {}
    _p, _n, n_levels = h.tree_level(0)
    for lv in range(-1, n_levels):
        p, n, _ = h.tree_level(lv)
        out[lv] = torch.as_tensor(_Dev(p, n), device='cuda').cpu().numpy().copy()
    return out


def _program(precision, n_in, seed):
    """A rotated, checkpointed last pass over an entangled 2^n_in-amplitude input (M = 6 / 5: the widest image count
    per warp store; the sums do not depend on M)."""
    M = 6 if precision == 'single' else 5
    n = n_in + M
    p = Prog(np.random.RandomState(seed), n).init(n_in)
    p.mux(n_in - 1, [0, n_in // 2])
    p.mux(1, [n_in - 1, 3])
    p.flag_last = True
    p.expand(M, [[0, 4], [1, 6], []] * 2)
    ops, tabs = p.finish()
    return n, ops, tabs


def _engine_child(res):
    for precision in ('single', 'double'):
        for n_in in N_INS:
            n, ops, tabs = _program(precision, n_in, 100 + n_in)
            with _native.Handle(n, precision) as h:
                h.run_program(ops, tabs)
                res['%s_%d:kern' % (precision, n_in)] = np.array(h.op_kernels()[-1])
                for lv, arr in _levels(h).items():
                    res['%s_%d:L%d' % (precision, n_in, lv)] = arr
                if precision == 'single' and n_in == N_INS[1]:
                    # the sampler's finer entries are pair sums of the written images' weights, even input first
                    res['single_amp'] = h.get_amplitudes()


def _q33_child(res):
    from qcmrf_b200 import B200Simulator, QCMRF, workloads
    C, _ = workloads.named('q33')
    sim = B200Simulator(precision='single', seed=2024, small_batch=False)
    prep = sim.prepare(QCMRF(C, workloads.theta_for(C)))
    sim.execute(prep, 1000, seed=1, stream=0)
    res['kern'] = np.array(sim.op_kernels()[-1])
    for lv, arr in _levels(sim._handle(prep.plan.n_phys, 'single')).items():
        res['L%d' % lv] = arr
    sim.close()


def _sums_name(shape, precision):
    if precision == 'double' and shape == '8x8':
        shape = '4x7'                                           # complex128's default shape
    w, tb = (int(v) for v in shape.split('x'))
    return 'k_expand_low_sums<%s,TB=%d,NW=%d>' % ('float,2' if precision == 'single' else 'double,1', tb, w)


def _spawn(tmp_path, what, mode, shape=None):
    out = str(tmp_path / ('%s_%s_%s.npz' % (what, mode, shape)))
    env = {k: v for k, v in os.environ.items() if not k.startswith('QCM_')}
    env['QCM_VIRTUAL_LAST'] = mode
    if shape:
        env['QCM_LOW_SHAPE'] = shape
    r = subprocess.run([sys.executable, os.path.abspath(__file__), out, what], env=env, timeout=1800,
                       capture_output=True, text=True)
    assert r.returncode == 0, (what, mode, shape, r.stdout[-2000:], r.stderr[-3000:])
    return dict(np.load(out))


@pytest.mark.parametrize('shape', SHAPES)
def test_virtual_sums_equal_the_materialising_tree(tmp_path, shape):
    ref = _spawn(tmp_path, 'engine', '0', shape)
    got = _spawn(tmp_path, 'engine', '1', shape)
    assert sorted(got) == sorted(ref)
    for key in ref:
        if key.endswith(':kern'):
            assert str(ref[key]).startswith('k_expand_low<'), (key, ref[key])
            assert str(got[key]) == _sums_name(shape, key.split('_')[0]), (key, got[key])
            continue
        assert np.array_equal(got[key], ref[key]), key
    for precision in ('single', 'double'):
        for n_in in N_INS:
            l0 = ref['%s_%d:L0' % (precision, n_in)]
            assert l0.dtype == np.float64 and l0.size == 1 << (n_in - 10) and (l0 > 0).all(), (precision, n_in)
            fine = ref['%s_%d:L-1' % (precision, n_in)]
            assert fine.size == 1 << (n_in - (1 if precision == 'single' else 0)), (precision, n_in)
    # complex64's finer level: entry p weighs input pair (2p, 2p + 1), i.e. all images of both inputs (logical index
    # x | image << n_in); the written images give it to fp32 rounding
    n_in = N_INS[1]
    img = (np.abs(ref['single_amp'].astype(np.complex128)) ** 2).reshape(-1, 1 << n_in).sum(axis=0)
    assert np.allclose(got['single_%d:L-1' % n_in], img[0::2] + img[1::2], rtol=1e-4, atol=0)


def test_q33_virtual_sums_equal_the_materialising_tree(tmp_path):
    import torch
    free, _ = torch.cuda.mem_get_info()
    if free < (70 << 30):                                       # the written reference: 64 GiB of state + input + tree
        pytest.skip('needs 70 GiB of free device memory')
    ref = _spawn(tmp_path, 'q33', '0')
    got = _spawn(tmp_path, 'q33', '1')
    assert str(ref['kern']).startswith('k_expand_low<') and str(got['kern']) == 'k_expand_low_sums<float,2,TB=8,NW=8>'
    assert sorted(got) == sorted(ref) and len(ref) > 3
    for key in ref:
        if key != 'kern':
            assert np.array_equal(got[key], ref[key]), key


if __name__ == '__main__':
    res = {}
    {'engine': _engine_child, 'q33': _q33_child}[sys.argv[2]](res)
    np.savez(sys.argv[1], **res)
