"""The virtual last pass (QCM_VIRTUAL_LAST): a rotated last expansion whose result is left unwritten, its images
computed by the readers from the pass's input with the kernel's own arithmetic.

Child processes run one corpus with the result always written (=0), always virtual (=1) and under the default size
rule (virtual above 2^30 amplitudes).  Everything the engine returns must be bit-identical between them: sampled keys
with and without a clbit map, the prefix post-selection (computed images), the general post-selection, the
amplitudes, the tree total and sharded device sampling (written out on demand), and whatever follows a dropped
descriptor (a next program, set_amplitudes, a rebuilt tree).
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

import engine_emulator as em                                # noqa: E402
from qcmrf_b200 import _native, fusion                      # noqa: E402
from test_engine_paths import Prog, TOL_AMP, _plan, _has_cuda   # noqa: E402

F = fusion
SHOTS = 4000
N_GLOBAL, RANK = 2, 3                                       # sharded cases: both global qubits are 1 on this rank
RANK_MASSES = [0.6, 0.3, 0.8]                               # the other ranks' masses (this rank's is its own)

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not _has_cuda(), reason='needs a CUDA device')]


def _cases():
    """(name, precision, n_local, sharded, ops, tabs): rotated last passes of every width, with and without
    diagonal members, with index qubit 0, and with global index qubits on a sharded handle."""
    rng = np.random.RandomState(11)
    out = []
    n_in = 11
    for precision, widths in (('single', (6, 7, 8)), ('double', (5, 6, 7, 8))):
        for M in widths:
            for n_diag in (0, 2):
                n = n_in + M
                p = Prog(rng, n).init(n_in)
                p.mux(3, [0, 5])                             # an entangled input
                ctrls = [[0, 4], [j % n_in for j in (1, 6)], []] * 3
                p.flag_last = True
                p.expand(M, ctrls[:M], n_diag=n_diag, diag_ctrl=[0, 7] if n_diag else ())
                ops, tabs = p.finish()
                out.append(('%s_M%d_diag%d' % (precision, M, n_diag), precision, n, False, ops, tabs))
        M = 7 if precision == 'single' else 6
        n = n_in + M
        for n_diag in (0, 1):
            p = Prog(rng, n).init(n_in)
            p.mux(2, [n + 1, 0])
            p.flag_last = True
            p.expand(M, [[n + 1, 0]] + [[n, j] for j in range(1, M)], n_diag=n_diag, diag_ctrl=[n + 1, 3])
            ops, tabs = p.finish()
            out.append(('%s_sharded_diag%d' % (precision, n_diag), precision, n, True, ops, tabs))
    return out


def _in_place_program(n, n_in, M, seed):
    """A program of the same size whose last pass is written in place (no flags)."""
    p = Prog(np.random.RandomState(seed), n).init(n_in)
    p.expand(M, [[0, 2]] + [[j] for j in range(1, M)])
    return p.finish()


def _dev(t, n, dtype):
    return t.zeros(n, dtype=dtype, device='cuda')


def _corpus_child(res):
    import torch as t
    for name, precision, n, sharded, ops, tabs in _cases():
        cl = list(range(n - 1, -1, -2)) + [-1, 0]
        with _native.Handle(n, precision) as h:
            if sharded:
                h.set_shard(N_GLOBAL, RANK)

            def sample(seed, stream, clbits=None):
                if not sharded:
                    return h.sample(SHOTS, seed, stream, clbit_qubit=clbits)
                masses = RANK_MASSES + [h.sample_prepare()]
                keys, mine = h.sample_sharded(SHOTS, seed, stream, masses, clbit_qubit=clbits)
                return np.where(mine, keys, np.uint64(0))

            gbits = (1 << n) if sharded else 0                  # a global bit in the masks (this rank's value)
            h.run_program(ops, tabs)
            res[name + ':kern'] = np.array(h.op_kernels())
            res[name + ':keys'] = sample(7, 1)
            res[name + ':keys_cl'] = sample(7, 2, cl)
            probs, kept = h.postselect((((1 << n) - 1) & ~63) | gbits, gbits, 6)
            res[name + ':pre'], res[name + ':pre_kept'] = probs, np.array(kept)
            tot = _dev(t, 1, t.float64)
            kd, md = _dev(t, SHOTS, t.int64), _dev(t, SHOTS, t.uint8)
            pd, kpd = _dev(t, 64, t.float64), _dev(t, 1, t.float64)
            t.cuda.synchronize()
            h.tree_total_device(tot.data_ptr())
            h.postselect_device((((1 << n) - 1) & ~63) | gbits, gbits, 6, pd.data_ptr(), kpd.data_ptr())
            if sharded:
                h.sample_sharded_device(SHOTS, 5, 3, RANK_MASSES + [h.sample_prepare()], cl, kd.data_ptr(), md.data_ptr())
            h.synchronize()
            res[name + ':total_dev'] = tot.cpu().numpy()
            res[name + ':pre_dev'] = pd.cpu().numpy()
            res[name + ':pre_kept_dev'] = kpd.cpu().numpy()
            if sharded:
                res[name + ':keys_dev'] = kd.cpu().numpy() * md.cpu().numpy()
            # general mask: the result is written out first; the tree stays and now reads the written images
            probs, kept = h.postselect((1 << (n - 1)) | 2 | gbits, 2 | gbits, 5)
            res[name + ':gen'], res[name + ':gen_kept'] = probs, np.array(kept)
            res[name + ':keys_after'] = sample(7, 1)
            res[name + ':amp'] = h.get_amplitudes()
            # each on-demand reader straight after a run
            h.run_program(ops, tabs)
            res[name + ':amp_first'] = h.get_amplitudes()
            h.run_program(ops, tabs)
            h.state_ptr()
            res[name + ':keys_state_ptr'] = sample(7, 1)
            h.run_program(ops, tabs)
            h.set_active(n)                                      # same width: the tree is dropped and rebuilt from the state
            res[name + ':keys_rebuilt'] = sample(7, 1)
            if sharded:
                continue
            # the unwritten result is dropped by a next program and by set_amplitudes; without the checkpoint flag the
            # sampler rebuilds the tree from the written-out result
            n_in = int(ops[0]['n_active_out'])
            ops2, tabs2 = _in_place_program(n, n_in, n - n_in, 99)
            h.run_program(ops, tabs)
            h.run_program(ops2, tabs2)
            res[name + ':next_amp'] = h.get_amplitudes()
            res[name + ':next_keys'] = sample(7, 1)
            h.run_program(ops, tabs)
            amps = np.random.RandomState(5).randn(1 << n) + 1j * np.random.RandomState(6).randn(1 << n)
            h.set_amplitudes(amps / np.linalg.norm(amps))
            res[name + ':set_amp'] = h.get_amplitudes()
            res[name + ':set_keys'] = sample(7, 1)
            ops3 = ops.copy()
            ops3[int(np.flatnonzero(ops3['flags'])[0])]['flags'] = F.QCM_FLAG_ROTATED_OUTPUT_OK
            h.run_program(ops3, tabs)
            res[name + ':nockpt_keys'] = sample(7, 1)


def _pipeline_child(res):
    """A pipelined run(list) against blocking runs of the same circuits (rotated last pass of 8 qubits on 13)."""
    from qcmrf_b200 import B200Simulator, QCMRF, workloads
    C = workloads.random_tree(11, 0, seed=3)
    circs = [QCMRF(C, workloads.theta_for(C, seed=10 + k)) for k in range(3)]
    sim = B200Simulator(precision='single', seed=5, small_batch=False, sweep_batch=False)
    r = sim.run(circs, shots=3000).result()
    res['pipe_kern'] = np.array(sim.op_kernels())
    for i, c in enumerate(circs):
        one = sim.run(c, shots=3000, stream_ids=[i]).result()
        for tag, rr, k in (('list', r, i), ('one', one, 0)):
            p, d = rr.postselected_probabilities(k)
            cnt = rr.get_counts(k)
            res['pipe%d_%s_pmf' % (i, tag)] = np.asarray(p)
            res['pipe%d_%s_delta' % (i, tag)] = np.array(d)
            res['pipe%d_%s_counts' % (i, tag)] = np.array(sorted((int(kk, 2), v) for kk, v in cnt.items()))
    sim.close()


def _large_child(res):
    """q33 (32 stored qubits, complex64: 2^32 amplitudes)."""
    from qcmrf_b200 import B200Simulator, QCMRF, workloads
    C, _ = workloads.named('q33')
    th = workloads.theta_for(C)
    sim = B200Simulator(precision='single', seed=2024, small_batch=False)
    r = sim.run(QCMRF(C, th), shots=20000).result()
    p, d = r.postselected_probabilities()
    res['pmf'], res['delta'] = np.asarray(p), np.array(d)
    res['counts'] = np.array(sorted((int(k, 2), v) for k, v in r.get_counts().items()))
    res['kern'] = np.array(sim.op_kernels())
    res['written'] = np.array([w for _k, _ms, _r, w in sim.op_profile()], dtype=np.uint64)
    sim.close()


def _spawn(tmp_path, what, mode):
    out = str(tmp_path / ('%s_%s.npz' % (what, mode)))
    env = {k: v for k, v in os.environ.items() if not k.startswith('QCM_')}
    if mode != 'unset':
        env['QCM_VIRTUAL_LAST'] = mode
    r = subprocess.run([sys.executable, os.path.abspath(__file__), out, what], env=env, timeout=900, capture_output=True, text=True)
    assert r.returncode == 0, (what, mode, r.stdout[-2000:], r.stderr[-3000:])
    return dict(np.load(out))


def test_virtual_readers_are_bit_identical_to_the_written_result(tmp_path):
    got = {m: _spawn(tmp_path, 'corpus', m) for m in ('0', '1', 'unset')}
    names = set(k.split(':')[0] for k in got['0'])
    assert len(names) == len(_cases())
    for key in got['0']:
        if key.endswith(':kern'):
            continue
        if key.endswith(':gen'):
            # the general post-selection adds into its pmf with fp64 atomics: the order of the additions varies
            assert np.allclose(got['1'][key], got['0'][key], rtol=1e-12, atol=0), key
            assert np.allclose(got['unset'][key], got['0'][key], rtol=1e-12, atol=0), key
            continue
        assert np.array_equal(got['1'][key], got['0'][key]), key
        assert np.array_equal(got['unset'][key], got['0'][key]), key        # all below 2^30 amplitudes: written
    for name, precision, n, sharded, ops, tabs in _cases():
        k0, k1, ku = (list(got[m][name + ':kern']) for m in ('0', '1', 'unset'))
        assert k0[-1].startswith('k_expand_low<') and ku == k0, (name, k0, ku)
        # diagonal members: no checkpoint (the pass need not preserve the norm), so no sums to compute and no launch
        assert k1[-1] == ('k_expand_low_sums<float,2,TB=8,NW=8>' if precision == 'single' else
                          'k_expand_low_sums<double,1,TB=7,NW=4>') if name.endswith('diag0') else k1[-1] == '', (name, k1)
        assert k1[:-1] == k0[:-1], (name, k1)
        assert len(np.unique(got['1'][name + ':keys'])) > 100
        if not sharded:
            want = em.run_plan(_plan(ops, tabs, n))[0]
            assert np.abs(got['1'][name + ':amp'] - want).max() < TOL_AMP[precision], name
            w = np.abs(want) ** 2
            assert np.isclose(float(got['1'][name + ':pre_kept']), w[:64].sum(), rtol=1e-4), name
            assert (w[got['1'][name + ':keys'].astype(np.int64)] > 0).all(), name
        assert np.array_equal(got['1'][name + ':keys_after'], got['1'][name + ':keys'])
        assert np.array_equal(got['1'][name + ':amp_first'], got['1'][name + ':amp'])


def test_pipelined_list_under_the_virtual_pass_equals_blocking_runs(tmp_path):
    got = _spawn(tmp_path, 'pipeline', '1')
    assert got['pipe_kern'][-1].startswith('k_expand_low_sums<'), got['pipe_kern']
    for i in range(3):
        for part in ('pmf', 'delta', 'counts'):
            assert np.array_equal(got['pipe%d_list_%s' % (i, part)], got['pipe%d_one_%s' % (i, part)]), (i, part)


def test_state_above_2_to_30_amplitudes_is_virtual_by_default(tmp_path):
    import torch
    free, _ = torch.cuda.mem_get_info()
    if free < (40 << 30):
        pytest.skip('needs 40 GiB of free device memory')
    ref = _spawn(tmp_path, 'large', '0')
    got = _spawn(tmp_path, 'large', 'unset')
    for part in ('pmf', 'delta', 'counts'):
        assert np.array_equal(got[part], ref[part]), part
    assert ref['kern'][-1].startswith('k_expand_low<'), ref['kern']
    assert got['kern'][-1].startswith('k_expand_low_sums<'), got['kern']
    assert int(got['written'].sum()) < (1 << 30), got['written']
    assert int(ref['written'].sum()) > (32 << 30)


if __name__ == '__main__':
    res = {}
    {'corpus': _corpus_child, 'pipeline': _pipeline_child, 'large': _large_child}[sys.argv[2]](res)
    np.savez(sys.argv[1], **res)
