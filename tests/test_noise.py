"""Noisy shots: Pauli gate errors as per-shot trajectories (qcm_run_noisy_small, k_traj) and readout errors
(k_readout_keys), from the public NoiseModel down to the kernels.

CPU: the model's validation, the density-matrix oracle (tests/density_oracle.py) against oracle.statevector, and
the encoded gate stream executed in numpy against both.  GPU: sampled key histograms against the density-matrix law,
exact cases bit for bit, reproducibility, the CTA-per-trajectory branch and the reference's transpiled flow (all 70
circuits of a scale)."""
import numpy as np
import pytest

import density_oracle as dm
from conftest import has_cuda
from oracle import statevector as sv
from qcmrf_b200 import QCMRF, B200Simulator, _native, ir, transpile
from qcmrf_b200.noise import NoiseModel, ReadoutError, depolarizing_error, encode, pauli_error


def gpu(test):
    return pytest.mark.gpu(pytest.mark.skipif(not has_cuda(), reason='needs a CUDA device')(test))


_FIXED_1Q = ('h', 'x', 'y', 'z', 's', 'sdg', 't', 'tdg', 'sx', 'sxdg', 'id')


def random_program(rng, N, n_gates, measured=None):
    """Random program over the ir gate surface that oracle.statevector also executes."""
    p = ir.Program(N, N)
    for _ in range(n_gates):
        r = rng.randint(7) if N > 1 else rng.randint(2)
        q = rng.permutation(N)
        if r == 0:
            p.gates.append(ir.Gate(_FIXED_1Q[rng.randint(len(_FIXED_1Q))], (int(q[0]),)))
        elif r == 1:
            p.gates.append(ir.Gate(['rz', 'rx', 'ry', 'p'][rng.randint(4)], (int(q[0]),), (float(rng.uniform(-3, 3)),)))
        elif r == 2:
            p.gates.append(ir.Gate('cx', (int(q[0]), int(q[1])), (), (1,)))
        elif r == 3:
            p.gates.append(ir.Gate('cz', (int(q[0]), int(q[1])), (), (1,)))
        elif r == 4:
            p.gates.append(ir.Gate('cp', (int(q[0]), int(q[1])), (float(rng.uniform(-3, 3)),), (1,)))
        else:
            k = rng.randint(1, N)
            cv = tuple(int(v) for v in rng.randint(0, 2, size=k))
            name = 'mcx' if r == 5 else 'mcp'
            params = (float(rng.uniform(-3, 3)),) if name == 'mcp' else ()
            p.gates.append(ir.Gate(name, tuple(int(x) for x in q[:k + 1]), params, cv))
    for c in (range(N) if measured is None else measured):
        p.measures[c] = c
    return p


def sv_probs(prog):
    psi, _ = sv.run_program(ir.to_oracle_ops(prog), prog.n_qubits)
    return np.abs(psi) ** 2


def reference_noise(N):
    """1- and 2-qubit depolarizing and Pauli errors, with a qubit-specific override and per-qubit readout."""
    nm = NoiseModel()
    nm.add_all_qubit_quantum_error(depolarizing_error(0.06, 1), ['sx', 'x', 'h', 'ry'])
    nm.add_all_qubit_quantum_error(pauli_error([('X', 0.04), ('Y', 0.03), ('Z', 0.05), ('I', 0.88)]), ['rz', 'rx', 's', 't'])
    nm.add_all_qubit_quantum_error(depolarizing_error(0.08, 2), ['cx'])
    nm.add_all_qubit_quantum_error(pauli_error([('IX', 0.05), ('ZY', 0.04), ('XI', 0.03), ('II', 0.88)]), ['cz', 'cp'])
    nm.add_quantum_error(pauli_error([('Y', 0.2), ('I', 0.8)]), ['sx', 'h'], [0])
    for q in range(N):
        nm.add_readout_error(ReadoutError([[1 - 0.01 * (q + 1), 0.01 * (q + 1)], [0.03 + 0.005 * q, 0.97 - 0.005 * q]]), [q])
    return nm


def transpiled_fixture(models, scale, graph, theta):
    C = models[scale]['GRAPHS'][graph]
    th = models[scale]['THETAS'][str(graph)][theta]
    return transpile([QCMRF(C, th)], basis_gates=['cx', 'id', 'rz', 'sx', 'x'])[0]


# ---------------------------------------------------------------------------------------------------- validation
def test_pauli_and_readout_errors_refuse_malformed_input():
    for bad in ([], [('XA', 1.0)], [('XYZ', 1.0)], [('X', 0.5), ('XI', 0.5)], [('X', -0.1), ('I', 1.1)],
                [('X', 0.5), ('I', 0.4)], [('x', 1.0)], [('X', float('nan'))]):
        with pytest.raises(ValueError):
            pauli_error(bad)
    pauli_error([('X', 0.5), ('I', 0.5 + 5e-13)])                     # within 1e-12 of 1
    for lam, n in ((-0.1, 1), (4 / 3 + 1e-9, 1), (16 / 15 + 1e-9, 2), (0.1, 3), (0.1, 1.5)):
        with pytest.raises(ValueError):
            depolarizing_error(lam, n)
    for bad in ([[0.9, 0.2], [0, 1]], [[1, 0]], [[1.1, -0.1], [0, 1]], [[0.5, 0.5], [0.5, 0.4]]):
        with pytest.raises(ValueError):
            ReadoutError(bad)


def test_depolarizing_error_has_aers_pauli_probabilities():
    for n, lam in ((1, 0.0), (1, 0.3), (1, 4 / 3), (2, 0.2), (2, 16 / 15)):
        d2 = 4 ** n
        e = depolarizing_error(lam, n)
        assert e.num_qubits == n and e.probs.size == d2
        assert e.probs[0] == pytest.approx(1 - lam * (d2 - 1) / d2, abs=1e-15)
        assert np.allclose(e.probs[1:], lam / d2, atol=1e-15, rtol=0)
    # lambda = 1: the uniform Pauli twirl; lambda = 4^n / (4^n - 1): no identity term
    assert np.allclose(depolarizing_error(1.0, 1).probs, 0.25) and np.allclose(depolarizing_error(1.0, 2).probs, 1 / 16)
    assert depolarizing_error(4 / 3, 1).probs[0] == 0


def test_pauli_labels_follow_qiskits_qubit_order():
    e = pauli_error([('XZ', 0.25), ('IY', 0.75)])
    assert dict(e.to_labels()) == {'XZ': 0.25, 'IY': 0.75}
    # 'IX' on cx acts on the control (the gate's first qubit): |00> -> cx -> X on qubit 0 -> |01> (qubit 0 set)
    p = ir.Program(2, 2, gates=[ir.Gate('cx', (0, 1), (), (1,))], measures={0: 0, 1: 1})
    nm = NoiseModel()
    nm.add_all_qubit_quantum_error(pauli_error([('IX', 1.0)]), ['cx'])
    assert np.allclose(dm.key_law(p, nm), [0, 1, 0, 0])


def test_noise_model_refusals():
    nm = NoiseModel()
    e1, e2 = depolarizing_error(0.1, 1), depolarizing_error(0.1, 2)
    for name in ('swap', 'measure', 'AND', 'ccx_composite', 'reset', 'barrier', 'toffoli'):
        with pytest.raises(ValueError):
            nm.add_all_qubit_quantum_error(e1, [name])
    with pytest.raises(ValueError):
        nm.add_all_qubit_quantum_error(e1, ['cx'])                     # a 1-qubit error on a 2-qubit gate
    with pytest.raises(ValueError):
        nm.add_all_qubit_quantum_error(e2, ['sx'])
    with pytest.raises(ValueError):
        nm.add_quantum_error(e2, ['cx'], [1, 1])
    with pytest.raises(ValueError):
        nm.add_quantum_error(e1, ['x'], [0, 1])
    with pytest.raises(ValueError):
        nm.add_all_qubit_quantum_error(np.eye(2), ['x'])               # only Pauli errors
    nm.add_all_qubit_quantum_error(e2, ['cnot'])                      # canonicalised to cx ...
    with pytest.raises(ValueError):
        nm.add_all_qubit_quantum_error(e2, ['cx'])                    # ... so this is a second error for cx
    nm.add_quantum_error(e2, ['cx'], [0, 1])
    with pytest.raises(ValueError):
        nm.add_quantum_error(e2, ['CX'], (0, 1))
    nm.add_quantum_error(e2, ['cx'], [1, 0])                          # another key
    ro = ReadoutError([[0.9, 0.1], [0.2, 0.8]])
    nm.add_all_qubit_readout_error(ro)
    with pytest.raises(ValueError):
        nm.add_all_qubit_readout_error(ro)
    nm.add_readout_error(ro, [3])
    for q in ([3], [0, 1], []):
        with pytest.raises(ValueError):
            nm.add_readout_error(ro, q)
    # an error attached to a gate of 3 or more qubits: transpile first
    nm2 = NoiseModel()
    nm2.add_all_qubit_quantum_error(e2, ['mcx'])
    p = ir.Program(3, 3, gates=[ir.Gate('mcx', (0, 1, 2), (), (1, 1))])
    with pytest.raises(ValueError, match='transpile first'):
        encode(p, nm2)
    encode(ir.Program(3, 3, gates=[ir.Gate('mcx', (0, 2), (), (1,))]), nm2)     # two qubits: fine


def test_noisy_circuit_above_the_small_limit_is_refused_before_any_launch(native_built):
    nm = NoiseModel()
    nm.add_all_qubit_quantum_error(depolarizing_error(0.1, 1), ['x'])
    big = ir.Program(14, 14, gates=[ir.Gate('x', (13,))], measures={13: 13})
    small = ir.Program(2, 2, gates=[ir.Gate('x', (0,))], measures={0: 0})
    with pytest.raises(ValueError, match='at most 13 qubits'):
        B200Simulator(noise_model=nm).run([small, big], shots=10)
    nm_ro = NoiseModel()
    nm_ro.add_readout_error(ReadoutError([[0.9, 0.1], [0, 1]]), [13])
    with pytest.raises(ValueError, match='at most 13 qubits'):
        B200Simulator().run(big, shots=10, noise_model=nm_ro)


def test_qubit_specific_error_wins_over_the_all_qubit_one():
    nm = NoiseModel()
    e_all, e_q1 = pauli_error([('X', 0.1), ('I', 0.9)]), pauli_error([('Z', 0.3), ('I', 0.7)])
    nm.add_all_qubit_quantum_error(e_all, ['x'])
    nm.add_quantum_error(e_q1, ['x'], [1])
    assert nm.gate_error('x', (1,)) is e_q1 and nm.gate_error('x', (0,)) is e_all and nm.gate_error('sx', (0,)) is None
    ro_all, ro_2 = ReadoutError([[0.9, 0.1], [0.1, 0.9]]), ReadoutError([[1, 0], [0.25, 0.75]])
    nm.add_readout_error(ro_2, [2])
    nm.add_all_qubit_readout_error(ro_all)
    assert nm.readout_error(2) is ro_2 and nm.readout_error(0) is ro_all
    p = ir.Program(3, 4, gates=[ir.Gate('x', (0,)), ir.Gate('x', (1,)), ir.Gate('x', (2,)), ir.Gate('x', (0,))],
                   measures={0: 0, 3: 2})
    e = encode(p, nm)
    cum = [e.cum[e.channel[i], :4] for i in range(4)]
    assert np.allclose(cum[0], np.cumsum(e_all.probs)) and np.allclose(cum[1], np.cumsum(e_q1.probs))
    assert np.allclose(cum[2], np.cumsum(e_all.probs))
    assert e.channel[0] == e.channel[3] and len(set(e.channel[:3])) == 3    # one record per (error, qubits)
    assert [list(e.chan_qubits[e.channel[i]]) for i in range(3)] == [[0, -1], [1, -1], [2, -1]]
    assert np.allclose(e.readout[0], [0.1, 0.1]) and np.allclose(e.readout[3], [0.0, 0.25])
    assert not e.readout[1:3].any() and not e.readout[4:].any()        # unmeasured clbits never flip


# -------------------------------------------------------------------------------------------------------- oracle
@pytest.mark.parametrize('N', [1, 2, 4, 6])
def test_density_oracle_without_noise_is_the_statevector_law(N):
    rng = np.random.RandomState(100 + N)
    for _ in range(4):
        p = random_program(rng, N, 30)
        rho = dm.run(p, NoiseModel())
        assert np.abs(np.real(np.diag(rho)) - sv_probs(p)).max() < 1e-14
        psi, _ = sv.run_program(ir.to_oracle_ops(p), N)
        assert np.abs(rho - np.outer(psi, psi.conj())).max() < 1e-13
        assert np.abs(dm.key_law(p) - sv.key_probabilities(psi, N, p.measures)).max() < 1e-14


def test_density_oracle_full_depolarizing_gives_the_maximally_mixed_state():
    nm = NoiseModel()
    nm.add_all_qubit_quantum_error(depolarizing_error(1.0, 1), ['h'])
    p = ir.Program(1, 1, gates=[ir.Gate('ry', (0,), (0.7,)), ir.Gate('h', (0,))], measures={0: 0})
    assert np.abs(dm.run(p, nm) - np.eye(2) / 2).max() < 1e-15
    # on one qubit of a Bell pair: the pair becomes I/4
    nm2 = NoiseModel()
    nm2.add_quantum_error(depolarizing_error(1.0, 1), ['sx'], [1])
    b = ir.Program(2, 2, gates=[ir.Gate('h', (0,)), ir.Gate('cx', (0, 1), (), (1,)), ir.Gate('sx', (1,))])
    assert np.abs(dm.run(b, nm2) - np.eye(4) / 4).max() < 1e-15


# ------------------------------------------------------------------------------------------------------ encoding
def apply_encoded_gate(e, g, psi):
    """Encoded gate g on psi: the 2x2 matrix on the target wherever (index & ctrl_mask) == ctrl_value."""
    psi = psi.copy()
    idx = np.arange(psi.size)
    t, cm, cv = int(e.target[g]), int(e.ctrl_mask[g]), int(e.ctrl_value[g])
    m = e.matrix[g, 0::2] + 1j * e.matrix[g, 1::2]
    i0 = idx[(((idx >> t) & 1) == 0) & ((idx & cm) == cv)]
    i1 = i0 | (1 << t)
    a0, a1 = psi[i0].copy(), psi[i1].copy()
    psi[i0], psi[i1] = m[0] * a0 + m[1] * a1, m[2] * a0 + m[3] * a1
    return psi


def run_encoded(e):
    """numpy executor of the ENCODED gate stream (no channels)."""
    psi = np.zeros(1 << e.n_qubits, dtype=np.complex128)
    psi[0] = 1
    for g in range(e.n_gates):
        psi = apply_encoded_gate(e, g, psi)
    return psi


def run_encoded_density(e):
    """The encoded stream with its channel records as a density-matrix map (Pauli k: code (k >> 2j) & 3 on
    chan_qubits[j]), against which the oracle checks what the kernel is handed."""
    N = e.n_qubits
    P = [np.eye(2), np.array([[0, 1], [1, 0]]), np.array([[0, -1j], [1j, 0]]), np.diag([1, -1])]

    def on(op, q):
        return np.kron(np.kron(np.eye(1 << (N - 1 - q)), op), np.eye(1 << q))

    rho = np.zeros((1 << N, 1 << N), dtype=np.complex128)
    rho[0, 0] = 1
    for g in range(e.n_gates):
        U = np.stack([apply_encoded_gate(e, g, col) for col in np.eye(1 << N, dtype=np.complex128)], axis=1)
        rho = U @ rho @ U.conj().T
        ch = int(e.channel[g])
        if ch >= 0:
            cum = e.cum[ch, :e.n_paulis[ch]]
            probs = np.diff(np.concatenate([[0.0], cum]))
            qs = [int(q) for q in e.chan_qubits[ch] if q >= 0]
            out = np.zeros_like(rho)
            for k, pk in enumerate(probs):
                A = np.eye(1 << N)
                for j, q in enumerate(qs):
                    A = on(P[(k >> (2 * j)) & 3], q) @ A
                out += pk * A @ rho @ A.conj().T
            rho = out
    return rho


@pytest.mark.parametrize('N', [1, 3, 5, 8])
def test_encoded_gate_stream_matches_the_statevector_oracle(N):
    rng = np.random.RandomState(7 + N)
    nm = reference_noise(N)
    for _ in range(5):
        p = random_program(rng, N, 40)
        e = encode(p, nm)
        assert e.n_gates == len(p.gates) and e.gate_noisy
        psi, _ = sv.run_program(ir.to_oracle_ops(p), N)
        assert np.abs(run_encoded(e) - psi).max() < 1e-12


def test_encoded_basis_programs_match_the_statevector_oracle(models):
    nm = reference_noise(10)
    for graph in range(7):
        T = transpiled_fixture(models, '0.25', graph, 3)
        p = ir.lower(T)
        assert isinstance(p, ir.BasisProgram)
        e = encode(p, nm)                                   # straight from the arrays (no Gate objects)
        assert p._gates is None
        psi, _ = sv.run_program(ir.to_oracle_ops(p), p.n_qubits)
        psi *= np.exp(1j * p.global_phase)
        got = run_encoded(e)
        ph = np.vdot(got, psi)                              # the engine drops the global phase
        assert abs(abs(ph) - 1) < 1e-10
        assert np.abs(got * ph / abs(ph) - psi).max() < 1e-10
        # the same program through its Gate list encodes to the same records
        g = encode(ir.Program(p.n_qubits, p.n_clbits, gates=list(p.gates), measures=dict(p.measures)), nm)
        for f in ('target', 'ctrl_mask', 'ctrl_value'):
            assert np.array_equal(getattr(e, f), getattr(g, f)), f
        assert np.abs(e.matrix - g.matrix).max() < 1e-15
        assert np.array_equal(e.channel >= 0, g.channel >= 0)
        on = e.channel >= 0                                  # channel records may be numbered differently
        assert np.array_equal(e.cum[e.channel[on]], g.cum[g.channel[on]])
        assert np.array_equal(e.chan_qubits[e.channel[on]], g.chan_qubits[g.channel[on]])


@pytest.mark.parametrize('N', [1, 2, 3, 4])
def test_encoded_channels_give_the_density_oracle_law(N):
    rng = np.random.RandomState(300 + N)
    nm = reference_noise(N)
    for _ in range(3):
        p = random_program(rng, N, 25)
        e = encode(p, nm)
        assert np.abs(run_encoded_density(e) - dm.run(p, nm)).max() < 1e-12


# ----------------------------------------------------------------------------------------------------------- GPU
def weissman_tv_bound(K, S, alpha=1e-6):
    """P(TV > bound) <= alpha for S draws over K outcomes (as tests/test_gpu_parity.py)."""
    return 0.5 * np.sqrt(2.0 * (K * np.log(2.0) + np.log(1.0 / alpha)) / S)


def counts_vec(counts, ncl):
    v = np.zeros(1 << ncl)
    for k, c in counts.items():
        v[int(k, 2)] = c
    return v


def assert_law(counts, law, shots, what, alpha=1e-6):
    ncl = int(np.log2(law.size))
    obs = counts_vec(counts, ncl)
    assert obs.sum() == shots, what
    assert obs[law <= 0].sum() == 0, what
    K = int((law > 0).sum())
    tv = 0.5 * np.abs(obs / shots - law).sum()
    assert tv < weissman_tv_bound(K, shots, alpha), (what, tv, weissman_tv_bound(K, shots, alpha))


@gpu
@pytest.mark.parametrize('precision', ['double', 'single'])
def test_noisy_counts_follow_the_density_matrix_law(models, precision):
    shots = 1 << 18
    rng = np.random.RandomState(2024)
    progs = [random_program(rng, N, 30, measured=range(N - 1) if N > 3 else None) for N in (2, 3, 4, 5, 6, 7)]
    progs += [ir.lower(transpiled_fixture(models, '0.25', g, 4)) for g in (0, 1, 2)]   # 3, 4 and 8 qubits
    nm = reference_noise(8)
    res = B200Simulator(precision=precision, seed=11, noise_model=nm).run(progs, shots=shots).result()
    for i, p in enumerate(progs):
        assert res.metadata(i)['noise'] and res.metadata(i)['path'] == 'noisy_trajectories'
        assert_law(res.get_counts(i), dm.key_law(p, nm), shots, (precision, i))


@gpu
@pytest.mark.parametrize('precision', ['double', 'single'])
def test_readout_only_noise_follows_its_law_on_the_ideal_kernel(precision):
    shots = 1 << 18
    rng = np.random.RandomState(5)
    progs = [random_program(rng, N, 25, measured=range(N - 1)) for N in (3, 5, 7)]
    nm = NoiseModel()
    for q in range(8):
        nm.add_readout_error(ReadoutError([[0.9 - 0.02 * q, 0.1 + 0.02 * q], [0.15, 0.85]]), [q])
    res = B200Simulator(precision=precision, seed=3, noise_model=nm).run(progs, shots=shots).result()
    for i, p in enumerate(progs):
        m = res.metadata(i)
        assert m['noise'] and m['path'] == 'batch_small'
        assert_law(res.get_counts(i), dm.key_law(p, nm), shots, (precision, i))


def _basis_state_circuit(N, ones, with_id):
    p = ir.Program(N, N + 1)
    for q in range(N):
        if q in ones:
            p.gates.append(ir.Gate('x', (q,)))
        p.gates.append(ir.Gate('id' if with_id else 'x', (q,)))
    for q in range(N):
        p.measures[q] = q                                   # clbit N is never measured: it stays '0'
    return p


@gpu
@pytest.mark.parametrize('precision', ['double', 'single'])
def test_certain_errors_give_exact_keys(precision):
    N, ones = 5, {1, 4}
    noisy, flipped = _basis_state_circuit(N, ones, True), _basis_state_circuit(N, ones, False)
    nm = NoiseModel()
    nm.add_all_qubit_quantum_error(pauli_error([('X', 1.0)]), ['id'])
    sim = B200Simulator(precision=precision, seed=42)
    got = sim.run(noisy, shots=5000, noise_model=nm).result()
    want = sim.run(flipped, shots=5000).result().get_counts()
    assert got.metadata()['path'] == 'noisy_trajectories'
    assert got.get_counts() == want and len(want) == 1
    # plus readout that always flips: the ideal key XOR the measured-bit mask, on the trajectory route
    mask = (1 << N) - 1
    nm.add_all_qubit_readout_error(ReadoutError([[0, 1], [1, 0]]))
    got = sim.run(noisy, shots=5000, noise_model=nm).result().get_counts()
    (key, cnt), = want.items()
    assert got == {format(int(key, 2) ^ mask, '0%db' % (N + 1)): cnt}


@gpu
@pytest.mark.parametrize('precision', ['double', 'single'])
def test_certain_readout_flips_are_the_ideal_keys_xor_the_measured_mask(precision):
    rng = np.random.RandomState(9)
    progs = [random_program(rng, N, 30, measured=[0, 2] + list(range(3, N))) for N in (3, 6, 9, 12)]
    nm = NoiseModel()
    nm.add_all_qubit_readout_error(ReadoutError([[0, 1], [1, 0]]))
    sim = B200Simulator(precision=precision, seed=77)
    got = sim.run(progs, shots=4096, noise_model=nm).result()
    ideal = sim.run(progs, shots=4096).result()
    for i, p in enumerate(progs):
        mask = sum(1 << c for c in p.measures)
        width = p.n_clbits
        assert got.get_counts(i) == {format(int(k, 2) ^ mask, '0%db' % width): v for k, v in ideal.get_counts(i).items()}
    # per shot, on the engine's keys: the readout launch flips exactly the measured bits of the ideal keys
    prs = [sim.prepare(p, small=True) for p in progs]
    args = ([pr.plan for pr in prs], [pr.clbit_map for pr in prs], [(0, 0, 0)] * len(prs), 4096, 77)
    ro = np.zeros((len(prs), 64, 2))
    for i, p in enumerate(progs):
        for c in p.measures:
            ro[i, c] = 1.0
    k0 = _native.run_batch_small(*args, precision=precision, stream_ids=[0, 1, 2, 3])[0]
    k1 = _native.run_batch_small(*args, precision=precision, stream_ids=[0, 1, 2, 3], readout=ro)[0]
    for i, p in enumerate(progs):
        assert np.array_equal(k1[i], k0[i] ^ np.uint64(sum(1 << c for c in p.measures)))


@gpu
@pytest.mark.parametrize('precision', ['double', 'single'])
def test_noisy_runs_are_reproducible_and_split_invariant(models, precision):
    rng = np.random.RandomState(1)
    progs = [random_program(rng, N, 20) for N in (2, 4, 11)] + [ir.lower(transpiled_fixture(models, '0.1', 2, 1))]
    ro_only = random_program(rng, 4, 10)
    nm = reference_noise(11)
    sim = B200Simulator(precision=precision, seed=123, noise_model=nm)
    circs = progs + [ro_only]
    a = sim.run(circs, shots=3000).result().get_counts()
    assert sim.run(circs, shots=3000).result().get_counts() == a
    b = sim.run(circs[:2], shots=3000, stream_ids=[0, 1]).result().get_counts() + \
        sim.run(circs[2:], shots=3000, stream_ids=[2, 3, 4]).result().get_counts()
    assert a == b
    assert sim.run(circs, shots=3000, seed=124).result().get_counts() != a
    # the model set through set_options, and overridden for one call
    sim2 = B200Simulator(precision=precision, seed=123)
    sim2.set_options(noise_model=nm)
    assert sim2.run(circs, shots=3000).result().get_counts() == a
    assert sim2.run(circs, shots=3000, noise_model=None).result().get_counts() == \
        B200Simulator(precision=precision, seed=123).run(circs, shots=3000).result().get_counts()


@gpu
@pytest.mark.parametrize('small_batch', [True, False])
def test_a_model_that_never_applies_is_no_model(models, small_batch):
    C = models['0.25']['GRAPHS'][2]
    th = models['0.25']['THETAS']['2'][0]
    circs = [QCMRF(C, th), transpiled_fixture(models, '0.25', 1, 0), QCMRF(models['0.5']['GRAPHS'][3], models['0.5']['THETAS']['3'][1])]
    unused = NoiseModel()
    unused.add_quantum_error(depolarizing_error(0.5, 1), ['x'], [40])             # no circuit has qubit 40
    unused.add_all_qubit_quantum_error(depolarizing_error(0.0, 2), ['cx'])       # identity only
    unused.add_readout_error(ReadoutError([[1, 0], [0, 1]]), [0])                # perfect readout
    ref = B200Simulator(seed=5, small_batch=small_batch).run(circs, shots=2000, n_vars=None).result()
    for nm in (NoiseModel(), unused):
        got = B200Simulator(seed=5, small_batch=small_batch, noise_model=nm).run(circs, shots=2000).result()
        assert got.get_counts() == ref.get_counts()
        for i in (0, 2):
            p, d = got.postselected_probabilities(i)
            q, e = ref.postselected_probabilities(i)
            assert np.array_equal(p, q) and d == e
            assert 'noise' not in got.metadata(i)


@gpu
def test_noisy_experiments_have_counts_and_no_exact_pmf(models):
    C = models['0.25']['GRAPHS'][1]
    th = models['0.25']['THETAS']['1'][0]
    nm_gate, nm_ro = NoiseModel(), NoiseModel()
    nm_gate.add_all_qubit_quantum_error(depolarizing_error(0.01, 2), ['cx'])
    nm_gate.add_all_qubit_quantum_error(depolarizing_error(0.01, 1), ['h'])          # the QCMRF's own gates
    nm_ro.add_all_qubit_readout_error(ReadoutError([[0.99, 0.01], [0.02, 0.98]]))
    T = transpiled_fixture(models, '0.25', 1, 0)
    for nm, path in ((nm_gate, 'noisy_trajectories'), (nm_ro, 'batch_small')):
        res = B200Simulator(seed=1, noise_model=nm).run([T, QCMRF(C, th)], shots=1000, n_vars=2).result()
        for i in range(2):
            assert sum(res.get_counts(i).values()) == 1000
            assert res.metadata(i)['noise'] is True
            with pytest.raises(ValueError):
                res.postselected_probabilities(i)
            with pytest.raises(ValueError):
                res.success_probability(i)
        assert res.metadata(0)['path'] == path
        assert res.to_dict()['results'][0]['success_probability'] is None


@gpu
@pytest.mark.parametrize('precision,N', [('single', 11), ('single', 12), ('single', 13), ('double', 11), ('double', 12),
                                         ('double', 13)])
def test_cta_per_trajectory_branch_per_qubit_marginals(precision, N):
    """Above 10 qubits a CTA runs one trajectory.  One-qubit gates with one-qubit errors factorise per qubit: each
    qubit's marginal is the 1-qubit density-matrix law of its own gates."""
    shots = 1 << 17
    rng = np.random.RandomState(N)
    p = ir.Program(N, N)
    for q in range(N):
        for _ in range(3):
            p.gates.append(ir.Gate('ry', (q,), (float(rng.uniform(0, np.pi)),)))
            name = ['sx', 'x', 'h', 'rz'][rng.randint(4)]
            p.gates.append(ir.Gate(name, (q,), (0.4,) if name == 'rz' else ()))
        p.measures[q] = q
    nm = NoiseModel()
    nm.add_all_qubit_quantum_error(depolarizing_error(0.2, 1), ['sx', 'h'])
    nm.add_all_qubit_quantum_error(pauli_error([('X', 0.1), ('Y', 0.05), ('I', 0.85)]), ['ry', 'x'])
    nm.add_quantum_error(pauli_error([('X', 0.5), ('I', 0.5)]), ['ry'], [N - 1])
    for q in range(0, N, 2):
        nm.add_readout_error(ReadoutError([[0.93, 0.07], [0.12, 0.88]]), [q])
    res = B200Simulator(precision=precision, seed=N, noise_model=nm).run(p, shots=shots).result()
    obs = np.zeros(N)
    for k, c in res.get_counts().items():
        bits = int(k, 2)
        for q in range(N):
            obs[q] += c * ((bits >> q) & 1)
    for q in range(N):
        sub = ir.Program(1, 1, gates=[ir.Gate(g.name, (0,), g.params) for g in p.gates if g.qubits == (q,)],
                         measures={0: 0})
        sub_nm = NoiseModel()
        for name in ('sx', 'h', 'ry', 'x'):
            e = nm.gate_error(name, (q,))
            if e is not None:
                sub_nm.add_all_qubit_quantum_error(e, [name])
        if nm.readout_error(q) is not None:
            sub_nm.add_all_qubit_readout_error(nm.readout_error(q))
        law = dm.key_law(sub, sub_nm)
        assert abs(obs[q] / shots - law[1]) < weissman_tv_bound(2, shots, 1e-6 / N), (q, obs[q] / shots, law[1])


@gpu
def test_reference_flow_under_noise(models):
    """The 70 transpiled fixture circuits of one scale in one run() call with depolarizing and readout noise."""
    shots = 1 << 17
    scale = '0.25'
    T = []
    for j in range(7):
        for i in range(10):
            T.append(transpiled_fixture(models, scale, j, i))
    nm = NoiseModel()
    nm.add_all_qubit_quantum_error(depolarizing_error(2e-3, 1), ['sx', 'x', 'id'])
    nm.add_all_qubit_quantum_error(depolarizing_error(2e-2, 2), ['cx'])
    nm.add_all_qubit_readout_error(ReadoutError([[0.98, 0.02], [0.03, 0.97]]))
    res = B200Simulator(seed=2025, noise_model=nm).run(T, shots=shots).result()
    counts = res.get_counts()
    assert len(counts) == 70
    checked = 0
    for i, t in enumerate(T):
        assert sum(counts[i].values()) == shots
        p = ir.lower(t)
        device = None if p.n_qubits <= dm.MAX_QUBITS else 'cuda'        # graph 3: 10 qubits, the torch backend
        assert_law(counts[i], dm.key_law(p, nm, device=device), shots, i, alpha=1e-6 / 70)
        checked += 1
    assert checked == 70
