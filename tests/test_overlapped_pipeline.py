"""The overlapped deferred pipeline of a plain handle: a circuit's sampler, post-selection and result copies run on a
reader stream beside the next circuit's program, each circuit on one of two buffer sets.

Child processes run lists of circuits with fresh theta through execute_deferred, three in flight, behind a device
sleep on the handle's stream so that the whole list is queued before the device reaches it (every reader then runs
beside the next program).  Keys, pmf and delta must be bit-identical to one blocking execute() per circuit, with the
last pass written (QCM_VIRTUAL_LAST=0) and left unwritten (=1), in both precisions and across a change of state size.
Readers that need the state (amplitudes, tree levels, a general-mask post-selection, a blocking execute) interleaved
with deferred circuits must return what they return in blocking order.  An engine built with both buffer sets as one
(QCM_TEST_ALIAS_SETS, the single set of the serial pipeline) must fail the list comparison.
"""
import collections
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
if __name__ == '__main__':                                   # child process: argv = [what, precision, engine library or '', shots]
    sys.path.insert(0, HERE)
    sys.path.insert(0, ROOT)
    if sys.argv[3]:                                          # before anything below loads the default library
        from qcmrf_b200 import _native
        _native.LIB_PATH = sys.argv[3]

from test_engine_paths import _has_cuda                      # noqa: E402

SHOTS = 3000
SLEEP_CYCLES = 200_000_000                                   # ~0.1 s on the handle's stream: the list queues behind it

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not _has_cuda(), reason='needs a CUDA device')]


def _items():
    """(cliques, theta) of a list with fresh theta per circuit and one change of state size in the middle."""
    from qcmrf_b200 import workloads
    small, large = workloads.random_tree(11, 0, seed=3), workloads.random_tree(12, 0, seed=4)
    return ([(small, workloads.theta_for(small, seed=s)) for s in range(10, 15)] +
            [(large, workloads.theta_for(large, seed=s)) for s in range(20, 24)])


def _sleep():
    import torch
    torch.cuda._sleep(SLEEP_CYCLES)                           # on the default stream, the handle's stream


def _same(a, b):
    return np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and a[2] == b[2]


def _child_list(precision, shots):
    """Pipelined list vs blocking calls; prints the indices of mismatching circuits."""
    from qcmrf_b200 import QCMRF, B200Simulator
    sim = B200Simulator(precision=precision, small_batch=False, sweep_batch=False, seed=77)
    prs = [sim.prepare(QCMRF(c, th)) for c, th in _items()]
    ref = [tuple(x.copy() if isinstance(x, np.ndarray) else x for x in sim.execute(pr, shots, seed=5, stream=i))
           for i, pr in enumerate(prs)]
    got = [None] * len(prs)
    fins = collections.deque()
    _sleep()
    for i, pr in enumerate(prs):
        if fins and (len(fins) == 3 or pr.plan.n_phys != prs[i - 1].plan.n_phys):
            if pr.plan.n_phys != prs[i - 1].plan.n_phys:
                while fins:                                   # a new state size replaces the handle: collect first
                    j, f = fins.popleft()
                    got[j] = f()
                _sleep()
            else:
                j, f = fins.popleft()
                got[j] = f()
        fins.append((i, sim.execute_deferred(pr, shots, seed=5, stream=i)))
    while fins:
        j, f = fins.popleft()
        got[j] = f()
    sim.close()
    bad = [i for i in range(len(prs)) if not _same(got[i], ref[i])]
    print(json.dumps({'bad': bad, 'n': len(prs)}))


def _child_readers(precision, shots):
    """Each reader that joins the streams, between deferred circuits, against the same sequence in blocking order."""
    import torch
    from test_virtual_sums import _levels
    from qcmrf_b200 import QCMRF, B200Simulator
    items = _items()[:5]

    def sequence(pipelined):
        sim = B200Simulator(precision=precision, small_batch=False, sweep_batch=False, seed=77)
        prs = [sim.prepare(QCMRF(c, th)) for c, th in items]
        n_phys = prs[0].plan.n_phys
        out, fins, done, general = [], [], [], []

        def run(i):
            if len(fins) == 3:                                # at most three in flight
                done.extend(fins.pop(0)())
            if pipelined:
                fins.append(sim.execute_deferred(prs[i], shots, seed=5, stream=i))
            else:
                fins.append(lambda r=sim.execute(prs[i], shots, seed=5, stream=i): r)
        _sleep()
        run(0)
        run(1)
        out.append(sim._handle(n_phys, precision).get_amplitudes(0, 1 << 12))
        run(2)
        h = sim._handle(n_phys, precision)
        h.sample_prepare()
        out.append(_levels(h)[0])
        run(3)
        probs, kept = sim._handle(n_phys, precision).postselect(1, 0, 4)     # a general mask: not the kept prefix
        out += [np.array([kept])]
        general.append(probs)
        out += [np.asarray(x) for x in sim.execute(prs[4], shots, seed=5, stream=4)]
        run(0)
        for f in fins:
            done.extend(f())
        out += [np.asarray(x) for x in done]
        torch.cuda.synchronize()
        sim.close()
        return out, general[0]

    (a, ga), (b, gb) = sequence(True), sequence(False)
    bad = [k for k in range(len(b)) if not np.array_equal(a[k], b[k])]
    # the general post-selection adds its bins with atomics: the order of those sums is not fixed, the values are
    if not np.allclose(ga, gb, rtol=1e-13, atol=0.0):
        bad.append('general')
    print(json.dumps({'bad': bad, 'n': len(b)}))


def _run_child(what, precision, virtual, lib=None, shots=SHOTS):
    env = dict(os.environ, QCM_VIRTUAL_LAST=str(virtual))
    code = ('import sys; sys.argv = %r; import runpy; ' % ['x', what, precision, lib or '', str(shots)] +
            'runpy.run_path(%r, run_name="__main__")' % os.path.abspath(__file__))
    r = subprocess.run([sys.executable, '-c', code], env=env, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize('virtual', [0, 1])
@pytest.mark.parametrize('precision', ['single', 'double'])
def test_pipelined_list_is_bit_identical_to_blocking_calls(precision, virtual):
    res = _run_child('list', precision, virtual)
    assert res['bad'] == [], res


@pytest.mark.parametrize('virtual', [0, 1])
@pytest.mark.parametrize('precision', ['single', 'double'])
def test_readers_between_deferred_circuits_see_blocking_order(precision, virtual):
    res = _run_child('readers', precision, virtual)
    assert res['bad'] == [], res


def _alias_build(dst):
    """The engine with QCM_TEST_ALIAS_SETS: the pipeline's two buffer sets are one, streams overlap as usual."""
    from qcmrf_b200 import build as b
    b.build_native()
    bdir = os.path.join(b.HERE, 'build')
    nvcc = b.shutil.which('nvcc') or '/usr/local/cuda/bin/nvcc'
    api = os.path.join(dst, 'qcm_api.o')
    subprocess.check_call([nvcc] + b.NVCC_FLAGS + ['-DQCM_TEST_ALIAS_SETS', '-I', os.path.join(ROOT, 'include'), '-I', b.CSRC,
                           '-c', os.path.join(b.CSRC, 'qcm_api.cu'), '-o', api])
    objs = [api] + [os.path.join(bdir, s.replace('.cu', '.o')) for s in b.SOURCES if s != 'qcm_api.cu']
    lib = os.path.join(dst, 'libqcmrf_b200.so')
    subprocess.check_call([nvcc, '-shared', '-o', lib] + objs + ['-gencode', 'arch=compute_100a,code=sm_100a', '-cudart', 'static'])
    return lib


def test_one_buffer_set_for_both_streams_is_detected():
    # enough shots that a circuit's sampler is still running when the next program overwrites a shared buffer
    shots = 500_000
    assert _run_child('list', 'single', 1, shots=shots)['bad'] == []
    with tempfile.TemporaryDirectory() as d:
        res = _run_child('list', 'single', 1, lib=_alias_build(d), shots=shots)
    assert res['bad'], 'overlapped readers on a shared buffer set went unnoticed'


if __name__ == '__main__':
    from qcmrf_b200 import _native
    assert _native.lib()._name == (sys.argv[3] or _native.LIB_PATH), _native.lib()._name
    {'list': _child_list, 'readers': _child_readers}[sys.argv[1]](sys.argv[2], int(sys.argv[4]))
