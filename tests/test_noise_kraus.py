"""Noisy shots with thermal relaxation, amplitude and phase damping, Kraus and coherent errors: the QuantumError
model, its encoding into error / Pauli / Kraus records, qcm_run_noisy_small_kraus and k_traj<R, CTA, true>.

The density-matrix law here never comes from noise.py's Kraus arrays: every error is built next to its expected
superoperator, written from the channel's closed form (or from the user's own operators), and composed / tensored
by hand.  CPU: the constructors, canonical Kraus forms, stage order, the encoded records executed as
superoperators, routing and the C ABI's refusals.  GPU: key histograms against the law, exact cases bit for bit,
renormalisation over 4000 gates, the CTA branch, reproducibility and routing, and the reference's transpiled flow
under a hardware-like model."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import density_oracle as dm
from conftest import has_cuda
from test_noise import (apply_encoded_gate, assert_law, random_program, run_encoded_density, transpiled_fixture,
                        weissman_tv_bound)
from qcmrf_b200 import B200Simulator, _native, ir
from qcmrf_b200 import noise as nz
from qcmrf_b200.noise import NoiseModel, ReadoutError, encode

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def gpu(test):
    return pytest.mark.gpu(pytest.mark.skipif(not has_cuda(), reason='needs a CUDA device')(test))


# ------------------------------------------------------------------------------------------ closed-form channels
# A 1-qubit superoperator acts on vec(rho) = (rho_00, rho_01, rho_10, rho_11); a 2-qubit one on the row-major vec of
# rho over (bit 1, bit 0), bit j the error's qubit j -- the density oracle's convention (kron(A, conj(A))).
def gad_super(a, p1, c):
    """rho_11 -> (1 - a) rho_11 + a p1 tr(rho), rho_01 -> c rho_01."""
    S = np.zeros((4, 4), dtype=np.complex128)
    S[0, 0], S[0, 3], S[3, 0], S[3, 3] = 1 - a * p1, a * (1 - p1), a * p1, 1 - a + a * p1
    S[1, 1] = S[2, 2] = c
    return S


def kraus_super(ops):
    return sum(np.kron(K, np.conj(K)) for K in ops)


def pauli_super(err):
    return sum(p * np.kron(dm._label_matrix(lab), dm._label_matrix(lab).conj()) for lab, p in err.to_labels())


def product_super(S0, S1):
    """S0 on qubit 0, S1 on qubit 1."""
    T = np.einsum('ABCD,EFGH->AEBFCGDH', S1.reshape(2, 2, 2, 2), S0.reshape(2, 2, 2, 2))
    return T.reshape(16, 16)


def AD(a, p1=0.0):
    return nz.amplitude_damping_error(a, p1), gad_super(a, p1, np.sqrt(1 - a))


def PD(b):
    return nz.phase_damping_error(b), gad_super(0, 0, np.sqrt(1 - b))


def PAD(a, b, p1=0.0):
    return nz.phase_amplitude_damping_error(a, b, p1), gad_super(a, p1, np.sqrt(1 - a - b))


def TR(t1, t2, time, p1=0.0):
    return nz.thermal_relaxation_error(t1, t2, time, p1), gad_super(1 - np.exp(-time / t1), p1, np.exp(-time / t2))


def KR(ops):
    return nz.kraus_error(ops), kraus_super([np.asarray(K, dtype=np.complex128) for K in ops])


def CU(U):
    return nz.coherent_unitary_error(U), kraus_super([np.asarray(U, dtype=np.complex128)])


def DEP(lam, n):
    e = nz.depolarizing_error(lam, n)
    return e, pauli_super(e)


def PAULI(terms):
    e = nz.pauli_error(terms)
    return e, pauli_super(e)


def compose(x, y):
    return x[0].compose(y[0]), y[1] @ x[1]


def expand(x, y):
    return x[0].expand(y[0]), product_super(x[1], y[1])


def tensor(x, y):
    return x[0].tensor(y[0]), product_super(y[1], x[1])


def rx(theta):
    c, s = np.cos(theta / 2), np.sin(theta / 2)
    return np.array([[c, -1j * s], [-1j * s, c]])


def user_gad_ops(a, p1):
    """Generalised amplitude damping as a user writes it: 4 textbook operators."""
    g0, g1 = np.sqrt(1 - p1), np.sqrt(p1)
    return [g0 * np.array([[1, 0], [0, np.sqrt(1 - a)]]), g0 * np.array([[0, np.sqrt(a)], [0, 0]]),
            g1 * np.array([[np.sqrt(1 - a), 0], [0, 1]]), g1 * np.array([[0, 0], [np.sqrt(a), 0]])]


class Model:
    """A NoiseModel with the expected superoperator of each of its errors."""

    def __init__(self):
        self.nm = NoiseModel()
        self.supers = {}

    def all(self, pair, names):
        self.supers[id(pair[0])] = pair[1]
        self.nm.add_all_qubit_quantum_error(pair[0], names)

    def local(self, pair, names, qubits):
        self.supers[id(pair[0])] = pair[1]
        self.nm.add_quantum_error(pair[0], names, qubits)


def law_rho(prog, model, device=None):
    """rho after the program: each gate U rho U^dagger, then its error's hand-built superoperator (numpy, or torch
    complex128 on `device`: the density oracle's two backends)."""
    N = prog.n_qubits
    T = dm.initial_state(N, device)
    cache = {}
    for g in prog.gates:
        err = dm._gate_error(model.nm, g)
        rows = [N - 1 - q for q in reversed(g.qubits)]
        cols = [2 * N - 1 - q for q in reversed(g.qubits)]
        if len(g.qubits) > 2:                               # no error: as the density oracle
            assert err is None
            T = dm.apply_controlled(T, g, N)
            continue
        key = (g.name, g.params, g.ctrl_values, len(g.qubits), id(err))
        S = cache.get(key)
        if S is None:
            U = g.matrix()
            S = np.kron(U, U.conj())
            if err is not None:
                S = model.supers[id(err)] @ S
            S = cache[key] = dm.operator(S, T)
        T = dm._apply(T, S, rows + cols)
    return T.reshape(1 << N, 1 << N)


def key_law(prog, model, device=None):
    return dm.key_law(prog, model.nm, rho=law_rho(prog, model, device))


def error_super(err, identity_kraus_at=()):
    """Superoperator of a QuantumError from its stages (the representation noise.py keeps); Kraus stages at the
    error's positions `identity_kraus_at` taken as the identity."""
    n = err.num_qubits
    S = np.eye(4 ** n, dtype=np.complex128)
    for st in err.stages:
        if st[0] == 'pauli':
            lab = nz.PauliError(len(st[2]), st[1])
            s1 = pauli_super(lab)
            if n == 2 and len(st[2]) == 1:
                s1 = product_super(s1, np.eye(4)) if st[2][0] == 0 else product_super(np.eye(4), s1)
        elif st[2] in identity_kraus_at:
            continue
        else:
            s1 = kraus_super(st[1])
            if n == 2:
                s1 = product_super(s1, np.eye(4)) if st[2] == 0 else product_super(np.eye(4), s1)
        S = s1 @ S
    return S


def random_rho(rng, d):
    A = rng.randn(d, d) + 1j * rng.randn(d, d)
    r = A @ A.conj().T
    return r / np.trace(r)


def random_cptp_ops(rng, n_ops):
    """n_ops Kraus operators of a random 1-qubit channel (the blocks of a random isometry)."""
    A = rng.randn(2 * n_ops, 2) + 1j * rng.randn(2 * n_ops, 2)
    Q, _ = np.linalg.qr(A)
    return [Q[2 * i:2 * i + 2] for i in range(n_ops)]


# ------------------------------------------------------------------------------------------------ constructors
def test_constructors_refuse_aers_out_of_range_parameters():
    bad = [lambda: nz.amplitude_damping_error(-0.1), lambda: nz.amplitude_damping_error(1.1),
           lambda: nz.amplitude_damping_error(0.1, -0.1), lambda: nz.amplitude_damping_error(0.1, 1.1),
           lambda: nz.amplitude_damping_error(float('nan')),
           lambda: nz.phase_damping_error(-0.1), lambda: nz.phase_damping_error(1.1),
           lambda: nz.phase_amplitude_damping_error(-0.1, 0.2), lambda: nz.phase_amplitude_damping_error(0.2, -0.1),
           lambda: nz.phase_amplitude_damping_error(0.6, 0.5), lambda: nz.phase_amplitude_damping_error(0.1, 0.1, 2),
           lambda: nz.thermal_relaxation_error(0, 1, 1), lambda: nz.thermal_relaxation_error(-1, 1, 1),
           lambda: nz.thermal_relaxation_error(1, 0, 1), lambda: nz.thermal_relaxation_error(1, -1, 1),
           lambda: nz.thermal_relaxation_error(1, 2 * (1 + 1e-12), 1), lambda: nz.thermal_relaxation_error(1, 1, -1e-9),
           lambda: nz.thermal_relaxation_error(1, 1, 1, 1.5), lambda: nz.thermal_relaxation_error(1, float('nan'), 1),
           lambda: nz.kraus_error([np.eye(3)]), lambda: nz.kraus_error([]), lambda: nz.kraus_error([[1, 0]]),
           lambda: nz.kraus_error([np.eye(2) * (1 + 1e-9)]), lambda: nz.kraus_error([np.array([[np.inf, 0], [0, 1]])]),
           lambda: nz.kraus_error([np.eye(2), np.eye(2)]),
           lambda: nz.coherent_unitary_error(np.diag([1, 1.001])), lambda: nz.coherent_unitary_error(np.eye(4)),
           lambda: nz.coherent_unitary_error([[1, 0]])]
    for f in bad:
        with pytest.raises(ValueError):
            f()
    # Aer's limits are accepted: t2 = 2 t1, infinite t1 / t2, a + b = 1, a sum of K^dagger K off by < 1e-10
    nz.thermal_relaxation_error(1, 2, 1)
    nz.thermal_relaxation_error(np.inf, np.inf, 1)
    nz.thermal_relaxation_error(np.inf, 5, 1)
    nz.phase_amplitude_damping_error(0.5, 0.5, 1)
    nz.kraus_error([np.eye(2) * (1 + 2e-11)])
    nz.coherent_unitary_error(rx(0.3))


@pytest.mark.parametrize('which', ['AD', 'PD', 'PAD', 'TR_T2_le_T1', 'TR_T2_gt_T1', 'TR_inf', 'KR', 'KR6', 'CU'])
def test_canonical_kraus_form_has_the_closed_form_action(which):
    rng = np.random.RandomState(hash(which) % 1000)
    pairs = {'AD': [AD(0.3), AD(0.7, 0.2), AD(1.0), AD(1.0, 1.0)], 'PD': [PD(0.4), PD(1.0)],
             'PAD': [PAD(0.2, 0.3, 0.1), PAD(0.5, 0.5), PAD(0.0, 0.9, 0.7)],
             'TR_T2_le_T1': [TR(50e-6, 30e-6, 8e-6), TR(1e-6, 1e-6, 1.0, 1.0), TR(40e-6, 10e-6, 3e-6, 0.3)],
             'TR_T2_gt_T1': [TR(20e-6, 35e-6, 6e-6, 0.05), TR(20e-6, 40e-6, 2e-6)],
             'TR_inf': [(nz.thermal_relaxation_error(np.inf, 30e-6, 5e-6), gad_super(0, 0, np.exp(-5 / 30)))],
             'KR': [KR(random_cptp_ops(rng, k)) for k in (1, 2, 3, 4)],
             'KR6': [KR(user_gad_ops(0.3, 0.2) + [np.zeros((2, 2))] * 2)],
             'CU': [CU(rx(0.7)), CU(np.diag([1, np.exp(0.4j)]))]}[which]
    for err, S in pairs:
        assert err.num_qubits == 1 and len(err.stages) == 1 and err.stages[0][0] == 'kraus'
        ops = err.stages[0][1]
        assert 1 <= len(ops) <= 4
        assert np.abs(sum(K.conj().T @ K for K in ops) - np.eye(2)).max() < 1e-12
        for _ in range(4):
            rho = random_rho(rng, 2)
            got = sum(K @ rho @ K.conj().T for K in ops)
            want = (S @ rho.reshape(-1)).reshape(2, 2)
            assert np.abs(got - want).max() < 1e-12, (which, err)


def test_generalised_amplitude_damping_from_six_textbook_operators_has_at_most_four():
    ops = user_gad_ops(0.4, 0.3)
    six = [ops[0], ops[1] * np.sqrt(0.5), ops[1] * np.sqrt(0.5), ops[2], ops[3] * np.sqrt(0.5), ops[3] * np.sqrt(0.5)]
    err = nz.kraus_error(six)
    assert len(err.stages[0][1]) == 4
    assert np.abs(error_super(err) - gad_super(0.4, 0.3, np.sqrt(0.6))).max() < 1e-12


def test_compose_tensor_and_expand_orders():
    rng = np.random.RandomState(3)
    a, b, c = AD(0.3, 0.1), CU(rx(0.9)), KR(random_cptp_ops(rng, 3))
    d2 = DEP(0.2, 2)
    cases = [compose(a, b), compose(b, a), compose(compose(a, b), c), tensor(a, b), expand(a, b), tensor(b, c),
             compose(d2, expand(a, c)), compose(tensor(b, a), d2), compose(DEP(0.1, 1), TR(50e-6, 40e-6, 9e-6)),
             expand(PAULI([('X', 0.3), ('I', 0.7)]), a)]
    for err, S in cases:
        assert np.abs(error_super(err) - S).max() < 1e-12, err
    # compose is not commutative here, and tensor / expand put their operands on different qubits
    assert np.abs(compose(a, b)[1] - compose(b, a)[1]).max() > 1e-3
    assert np.abs(tensor(a, b)[1] - expand(a, b)[1]).max() > 1e-3
    # an expanded error on cx: position 0 is the control (the gate's first qubit)
    m = Model()
    m.all(expand(AD(1.0), AD(0.0)), ['cx'])
    p = ir.Program(2, 2, gates=[ir.Gate('x', (0,)), ir.Gate('cx', (0, 1), (), (1,))], measures={0: 0, 1: 1})
    assert np.allclose(key_law(p, m), [0, 0, 1, 0])            # |11> -> control damped -> qubit 1 set only


def test_ideal_errors_and_models():
    for err in (nz.thermal_relaxation_error(50e-6, 30e-6, 0.0), nz.amplitude_damping_error(0),
                nz.phase_damping_error(0), nz.phase_amplitude_damping_error(0, 0, 0.3),
                nz.thermal_relaxation_error(np.inf, np.inf, 1.0), nz.coherent_unitary_error(np.eye(2)),
                nz.kraus_error([np.eye(2)]), nz.amplitude_damping_error(0).expand(nz.phase_damping_error(0)),
                nz.depolarizing_error(0, 1).compose(nz.amplitude_damping_error(0))):
        assert err.ideal(), err
    for err in (nz.amplitude_damping_error(1e-6), nz.thermal_relaxation_error(50e-6, 30e-6, 1e-9),
                nz.coherent_unitary_error(rx(1e-3)), nz.amplitude_damping_error(0).expand(nz.phase_damping_error(0.1)),
                nz.depolarizing_error(0.01, 1).compose(nz.amplitude_damping_error(0))):
        assert not err.ideal(), err
    nm = NoiseModel()
    nm.add_all_qubit_quantum_error(nz.thermal_relaxation_error(50e-6, 30e-6, 0.0), ['x', 'sx'])
    assert nm.is_ideal()
    nm.add_all_qubit_quantum_error(nz.thermal_relaxation_error(50e-6, 30e-6, 1e-8), ['id'])
    assert not nm.is_ideal()
    # an ideal error attaches no record
    e = encode(ir.Program(1, 1, gates=[ir.Gate('x', (0,)), ir.Gate('id', (0,))], measures={0: 0}), nm)
    assert list(e.channel) == [-1, 0] and e.kraus


def test_refusals_of_shape_and_stage_count():
    a, d2 = nz.amplitude_damping_error(0.1), nz.depolarizing_error(0.1, 2)
    with pytest.raises(ValueError, match='qubits'):
        d2.tensor(a)
    with pytest.raises(ValueError, match='qubits'):
        a.expand(d2)
    with pytest.raises(ValueError):
        a.expand(a).expand(a)
    with pytest.raises(ValueError):
        a.compose(d2)
    four = a.compose(a).compose(a).compose(a)
    assert len(four.stages) == 4
    with pytest.raises(ValueError, match='at most 4 stages'):
        four.compose(a)
    with pytest.raises(ValueError, match='at most 4 stages'):
        a.compose(a).compose(a).expand(a.compose(a))
    with pytest.raises(ValueError):
        a.compose(np.eye(2))
    # 2-qubit Kraus: a product of 1-qubit channels is accepted, anything else refused with the reason
    A, B = AD(0.3)[0].stages[0][1], random_cptp_ops(np.random.RandomState(1), 2)
    err = nz.kraus_error([np.kron(Bk, Ak) for Ak in A for Bk in B])          # A on qubit 0, B on qubit 1
    assert err.num_qubits == 2 and [st[0] for st in err.stages] == ['kraus', 'kraus']
    assert np.abs(error_super(err) - product_super(kraus_super(A), kraus_super(B))).max() < 1e-12
    cnot = np.eye(4)[[0, 3, 2, 1]]
    for ops in ([cnot], [np.sqrt(0.9) * np.eye(4), np.sqrt(0.1) * np.kron(dm._PAULI['X'], dm._PAULI['X'])]):
        with pytest.raises(ValueError, match='tensor products of 1-qubit ones'):
            nz.kraus_error(ops)


def test_noise_model_takes_quantum_errors_and_keeps_its_rules():
    nm = NoiseModel()
    t = nz.thermal_relaxation_error(50e-6, 30e-6, 1e-7)
    nm.add_all_qubit_quantum_error(t, ['x'])
    with pytest.raises(ValueError):
        nm.add_all_qubit_quantum_error(t, ['x'])                              # compose instead
    with pytest.raises(ValueError):
        nm.add_all_qubit_quantum_error(t, ['cx'])
    with pytest.raises(ValueError):
        nm.add_all_qubit_quantum_error(t.expand(t), ['sx'])
    nm.add_all_qubit_quantum_error(t.expand(t), ['cx'])
    for name in ('reset', 'measure', 'swap'):
        with pytest.raises(ValueError):
            nm.add_all_qubit_quantum_error(t, [name])
    with pytest.raises(ValueError):
        nm.add_all_qubit_quantum_error([np.eye(2)], ['sx'])
    assert isinstance(nz.depolarizing_error(0.1, 1), nz.QuantumError)
    assert isinstance(nz.pauli_error([('X', 1.0)]), nz.PauliError)


# -------------------------------------------------------------------------------------------------------- records
def run_records(e):
    """The encoded stream with its error records as a density-matrix map: stages in order, a Pauli stage from its
    cumulative table, a Kraus stage as sum_i K_i rho K_i^dagger of its recorded operators on its qubit."""
    if not e.kraus:
        return run_encoded_density(e)
    N = e.n_qubits
    P = [np.eye(2), dm._PAULI['X'], dm._PAULI['Y'], dm._PAULI['Z']]

    def on(op, q):
        return np.kron(np.kron(np.eye(1 << (N - 1 - q)), op), np.eye(1 << q))

    rho = np.zeros((1 << N, 1 << N), dtype=np.complex128)
    rho[0, 0] = 1
    for g in range(e.n_gates):
        U = np.stack([apply_encoded_gate(e, g, col) for col in np.eye(1 << N, dtype=np.complex128)], axis=1)
        rho = U @ rho @ U.conj().T
        k = int(e.channel[g])
        if k < 0:
            continue
        for j in range(int(e.err_n_stages[k])):
            idx = int(e.err_index[k, j])
            out = np.zeros_like(rho)
            if e.err_kind[k, j] == 0:
                probs = np.diff(np.concatenate([[0.0], e.cum[idx, :e.n_paulis[idx]]]))
                qs = [int(q) for q in e.chan_qubits[idx] if q >= 0]
                for kk, pk in enumerate(probs):
                    A = np.eye(1 << N)
                    for jj, q in enumerate(qs):
                        A = on(P[(kk >> (2 * jj)) & 3], q) @ A
                    out += pk * A @ rho @ A.conj().T
            else:
                ops = e.kraus_ops[idx, :e.kraus_n_ops[idx]]
                for K in ops:
                    A = on((K[0::2] + 1j * K[1::2]).reshape(2, 2), int(e.kraus_qubit[idx]))
                    out += A @ rho @ A.conj().T
            rho = out
    return rho


def mixed_model(N):
    """Every kind of error: damping with excited population, phase damping, thermal relaxation with T2 <= T1 and
    T1 < T2 <= 2 T1, user Kraus operators, a coherent unitary, depolarizing composed with relaxation, expand on cx,
    a 2-qubit Pauli error, a qubit-specific override and per-qubit readout."""
    m = Model()
    m.all(AD(0.15, 0.2), ['sx'])
    m.all(PD(0.3), ['h'])
    m.all(TR(50e-6, 30e-6, 8e-6), ['x', 'y'])
    m.all(TR(20e-6, 35e-6, 6e-6, 0.05), ['ry'])
    m.all(KR(user_gad_ops(0.2, 0.3)), ['rz'])
    m.all(CU(rx(0.35)), ['s', 'sdg'])
    m.all(compose(DEP(0.08, 1), TR(40e-6, 60e-6, 5e-6)), ['t', 'rx'])
    m.all(compose(DEP(0.06, 2), expand(TR(30e-6, 20e-6, 4e-6), AD(0.2, 0.1))), ['cx'])
    m.all(tensor(PD(0.25), PAD(0.1, 0.2)), ['cz'])
    m.all(PAULI([('IX', 0.05), ('ZY', 0.04), ('II', 0.91)]), ['cp'])
    m.local(compose(AD(0.5), CU(np.diag([1, 1j]))), ['sx', 'h'], [0])
    for q in range(N):
        m.nm.add_readout_error(ReadoutError([[1 - 0.01 * (q + 1), 0.01 * (q + 1)], [0.03 + 0.005 * q, 0.97 - 0.005 * q]]), [q])
    return m


def hardware_model():
    """tools/noise_bench.py's hardware-like model."""
    m = Model()
    m.all(compose(DEP(1e-3, 1), TR(100e-6, 80e-6, 35.5e-9)), ['sx', 'x', 'id'])
    t2q = TR(100e-6, 80e-6, 300e-9)
    m.all(compose(DEP(1e-2, 2), expand(t2q, t2q)), ['cx'])
    m.nm.add_all_qubit_readout_error(ReadoutError([[0.98, 0.02], [0.02, 0.98]]))
    return m


@pytest.mark.parametrize('N', [1, 2, 3, 4])
def test_encoded_records_give_the_closed_form_law(N):
    rng = np.random.RandomState(500 + N)
    m = mixed_model(N)
    for _ in range(3):
        p = random_program(rng, N, 25)
        e = encode(p, m.nm)
        if any(g.name in ('sx', 'h', 'x', 'y', 'ry', 'rz', 's', 'sdg', 't', 'rx', 'cx', 'cz') for g in p.gates):
            assert e.kraus
        assert np.abs(run_records(e) - law_rho(p, m)).max() < 1e-12


def test_encoded_basis_programs_give_the_closed_form_law(models):
    m = hardware_model()
    for graph in (0, 1):                                    # 3 and 4 qubits
        p = ir.lower(transpiled_fixture(models, '0.25', graph, 2))
        assert isinstance(p, ir.BasisProgram)
        e = encode(p, m.nm)
        assert p._gates is None and e.kraus
        g = encode(ir.Program(p.n_qubits, p.n_clbits, gates=list(p.gates), measures=dict(p.measures)), m.nm)
        assert np.array_equal(e.channel >= 0, g.channel >= 0)
        on = e.channel >= 0
        for f in ('err_n_stages', 'err_kind'):
            assert np.array_equal(getattr(e, f)[e.channel[on]], getattr(g, f)[g.channel[on]])
        rho = run_records(e)
        want = law_rho(ir.Program(p.n_qubits, p.n_clbits, gates=list(p.gates), measures=dict(p.measures)), m)
        assert np.abs(rho - want).max() < 1e-12
        assert np.abs(run_records(g) - want).max() < 1e-12


def test_pauli_only_models_keep_the_old_records_and_route():
    rng = np.random.RandomState(8)
    nm = NoiseModel()
    nm.add_all_qubit_quantum_error(nz.depolarizing_error(0.06, 1), ['sx', 'x', 'h'])
    nm.add_all_qubit_quantum_error(nz.pauli_error([('X', 0.1), ('I', 0.9)]), ['rz'])
    nm.add_all_qubit_quantum_error(nz.depolarizing_error(0.08, 2), ['cx'])
    p = random_program(rng, 4, 40)
    e = encode(p, nm)
    assert not e.kraus and e.gate_noisy
    n_err = len(e.err_n_stages)
    assert n_err == len(e.n_paulis)                          # error k is channel k: one Pauli stage each
    assert np.array_equal(e.err_n_stages, np.ones(n_err)) and not e.err_kind.any()
    assert np.array_equal(e.err_index[:, 0], np.arange(n_err)) and not len(e.kraus_n_ops)
    # the records of the old encoding: cumulative tables of the model's probabilities, on the gates' qubits
    for i, g in enumerate(p.gates):
        err = nm.gate_error(g.name, g.qubits)
        if err is None or len(g.qubits) > 2:
            assert e.channel[i] == -1
            continue
        c = e.channel[i]
        assert np.array_equal(e.cum[c, :err.probs.size - 1], np.cumsum(err.probs)[:-1])
        assert list(e.chan_qubits[c][:len(g.qubits)]) == list(g.qubits)
    # one composed error anywhere moves the circuit to the stage records
    nm.add_all_qubit_quantum_error(nz.depolarizing_error(0.01, 1).compose(nz.depolarizing_error(0.01, 1)), ['y'])
    p.gates.append(ir.Gate('y', (1,)))
    assert encode(p, nm).kraus


# ---------------------------------------------------------------------------------------------------------- C ABI
def _tiny_records():
    m = Model()
    m.all(compose(DEP(0.1, 1), AD(0.2)), ['x'])
    m.all(expand(AD(0.3), PD(0.2)), ['cx'])
    p = ir.Program(3, 3, gates=[ir.Gate('x', (0,)), ir.Gate('cx', (0, 2), (), (1,))], measures={0: 0, 2: 2})
    return _native._noisy_records([encode(p, m.nm)], True)


def _call(rec, shots=16, **over):
    nq, gb, gates, channels, errors, krauses, cq, ncl, ro = rec
    a = dict(errors=errors, n_errors=len(errors), channels=channels, n_channels=len(channels), krauses=krauses,
             n_kraus=len(krauses))
    a.update(over)
    keys = np.zeros(max(shots, 1), dtype=np.uint64)
    ptr = lambda x: None if x is None else x.ctypes.data
    return _native.lib().qcm_run_noisy_small_kraus(0, _native.QCM_C128, 1, ptr(nq), ptr(gb), ptr(gates), ptr(a['errors']),
                                                   a['n_errors'], ptr(a['channels']), a['n_channels'], ptr(a['krauses']),
                                                   a['n_kraus'], ptr(cq), ptr(ncl), None, None, shots, 1, ptr(keys), None)


def test_cabi_struct_layouts_match_the_header(tmp_path):
    src = r'''
    #include <stddef.h>
    #include <stdio.h>
    #include "qcmrf_b200.h"
    int main(void){ printf("%zu %zu %zu %zu %zu %zu", sizeof(qcm_kraus), offsetof(qcm_kraus, n_ops),
        offsetof(qcm_kraus, qubit), sizeof(qcm_gate_error), offsetof(qcm_gate_error, kind),
        offsetof(qcm_gate_error, index)); return 0; }
    '''
    exe = str(tmp_path / 'qcm_kraus_layout')
    subprocess.run(['gcc', '-x', 'c', '-', '-I', os.path.join(ROOT, 'include'), '-o', exe], input=src, text=True, check=True)
    vals = list(map(int, subprocess.run([exe], capture_output=True, text=True).stdout.split()))
    K, E = _native.KRAUS_DTYPE, _native.GATE_ERROR_DTYPE
    assert vals == [K.itemsize, K.fields['n_ops'][1], K.fields['qubit'][1], E.itemsize, E.fields['kind'][1],
                    E.fields['index'][1]]


def test_cabi_refuses_malformed_records_before_any_device_query(native_built):
    rec = _tiny_records()
    errors, krauses = rec[4], rec[5]
    assert 'qcm_run_noisy_small_kraus' in _native.SYMBOLS
    assert _call(rec, shots=0) == 0                          # well-formed; no shots: no device needed

    def bad(**over):
        assert _call(rec, **over) == -1, over                # QCM_ERR_INVALID, with or without a GPU

    def with_err(f):
        e = errors.copy()
        f(e)
        return e

    def with_kr(f):
        k = krauses.copy()
        f(k)
        return k

    bad(errors=None)
    bad(n_errors=-1)
    bad(errors=with_err(lambda e: e.__setitem__('n_stages', 0)))
    bad(errors=with_err(lambda e: e.__setitem__('n_stages', 5)))
    bad(errors=with_err(lambda e: e['kind'].__setitem__((0, 0), 2)))
    bad(errors=with_err(lambda e: e['index'].__setitem__((0, 1), len(krauses))))
    bad(errors=with_err(lambda e: e['index'].__setitem__((0, 0), len(rec[3]))))
    bad(errors=with_err(lambda e: e['index'].__setitem__((0, 0), -1)))
    bad(n_errors=len(errors) - 1)                            # a gate's error index out of range
    bad(n_kraus=0)
    bad(krauses=with_kr(lambda k: k['n_ops'].__setitem__(0, 0)))
    bad(krauses=with_kr(lambda k: k['n_ops'].__setitem__(0, 5)))
    bad(krauses=with_kr(lambda k: k['qubit'].__setitem__(0, -1)))
    bad(krauses=with_kr(lambda k: k['qubit'].__setitem__(0, 3)))    # not in [0, N)
    bad(krauses=with_kr(lambda k: k['qubit'].__setitem__(0, 1)))    # in range, but not one of the x gate's qubits
    bad(krauses=with_kr(lambda k: k['k'].__setitem__((0, 0, 0), np.nan)))
    bad(krauses=with_kr(lambda k: k['k'].__setitem__((0, 0, 0), k['k'][0, 0, 0] + 1e-9)))
    # within 1e-10 of trace preserving is accepted
    assert _call(rec, shots=0, krauses=with_kr(lambda k: k['k'].__setitem__((0, 0, 0), k['k'][0, 0, 0] + 1e-12))) == 0


@pytest.mark.skipif(has_cuda(), reason='this checks the GPU-less failure mode')
def test_cabi_well_formed_call_without_a_gpu_reports_no_device(native_built):
    assert _call(_tiny_records()) == -5                      # QCM_ERR_NO_DEVICE


# ----------------------------------------------------------------------------------------------------------- GPU
@gpu
@pytest.mark.parametrize('precision', ['double', 'single'])
def test_kraus_counts_follow_the_density_matrix_law(models, precision):
    shots = 1 << 18
    rng = np.random.RandomState(4242)
    progs = [random_program(rng, N, 30, measured=range(N - 1) if N > 3 else None) for N in (2, 3, 4, 5, 6, 7)]
    progs += [ir.lower(transpiled_fixture(models, '0.25', g, 4)) for g in (0, 1, 2)]   # 3, 4 and 8 qubits
    m = mixed_model(8)
    m.all(compose(DEP(1e-2, 1), TR(60e-6, 90e-6, 2e-6, 0.02)), ['id'])
    res = B200Simulator(precision=precision, seed=17, noise_model=m.nm).run(progs, shots=shots).result()
    for i, p in enumerate(progs):
        assert res.metadata(i)['noise'] and res.metadata(i)['path'] == 'noisy_trajectories_kraus', i
        if not isinstance(p, ir.BasisProgram):
            law = key_law(p, m)
        else:
            law = key_law(ir.Program(p.n_qubits, p.n_clbits, gates=list(p.gates), measures=dict(p.measures)), m)
        assert_law(res.get_counts(i), law, shots, (precision, i))


@gpu
@pytest.mark.parametrize('precision', ['double', 'single'])
def test_certain_damping_and_stage_order_give_exact_keys(precision):
    sim = B200Simulator(precision=precision, seed=9)
    N, shots = 6, 4096
    rng = np.random.RandomState(0)
    # amplitude damping 1 after x on every qubit: every shot reads all zeros
    p = ir.Program(N, N)
    for q in range(N):
        p.gates += [ir.Gate('ry', (q,), (float(rng.uniform(0, 3)),)), ir.Gate('x', (q,)), ir.Gate('h', (q,)),
                    ir.Gate('h', (q,))]
        p.measures[q] = q
    nm = NoiseModel()
    nm.add_all_qubit_quantum_error(nz.amplitude_damping_error(1.0), ['x'])
    r = sim.run(p, shots=shots, noise_model=nm).result()
    assert r.metadata()['path'] == 'noisy_trajectories_kraus' and r.get_counts() == {'0' * N: shots}
    # full relaxation to the excited state after id: all ones
    p = ir.Program(N, N, gates=[ir.Gate(n, (q,)) for q in range(N) for n in ('h', 'id')], measures={q: q for q in range(N)})
    nm = NoiseModel()
    nm.add_all_qubit_quantum_error(nz.thermal_relaxation_error(1e-6, 1e-6, 1.0, excited_state_population=1), ['id'])
    assert sim.run(p, shots=shots, noise_model=nm).result().get_counts() == {'1' * N: shots}
    # compose order: damping then X (as a Kraus operator) leaves |1>, X then damping leaves |0>
    X = nz.kraus_error([dm._PAULI['X']])
    p = ir.Program(1, 1, gates=[ir.Gate('x', (0,)), ir.Gate('id', (0,))], measures={0: 0})
    for err, key in ((nz.amplitude_damping_error(1.0).compose(X), '1'), (X.compose(nz.amplitude_damping_error(1.0)), '0')):
        nm = NoiseModel()
        nm.add_all_qubit_quantum_error(err, ['id'])
        assert sim.run(p, shots=shots, noise_model=nm).result().get_counts() == {key: shots}
    # expand on cx: position 0 is the control.  |11> with the control damped reads '10', the target damped '01'
    p = ir.Program(2, 2, gates=[ir.Gate('x', (0,)), ir.Gate('cx', (0, 1), (), (1,))], measures={0: 0, 1: 1})
    ad1, ad0 = nz.amplitude_damping_error(1.0), nz.amplitude_damping_error(0.0)
    for err, key in ((ad1.expand(ad0), '10'), (ad1.tensor(ad0), '01')):
        nm = NoiseModel()
        nm.add_all_qubit_quantum_error(err, ['cx'])
        assert sim.run(p, shots=shots, noise_model=nm).result().get_counts() == {key: shots}


@gpu
def test_long_circuit_with_weak_damping_stays_normalised():
    """4000 gates, weak amplitude damping after every one, complex64: every Kraus stage renormalises the state, so
    the law still holds and no trajectory's norm fails."""
    N, shots = 6, 1 << 18
    rng = np.random.RandomState(77)
    p = ir.Program(N, N)
    while len(p.gates) < 4000:
        q = rng.permutation(N)
        r = rng.randint(4)
        if r == 0:
            p.gates.append(ir.Gate('cx', (int(q[0]), int(q[1])), (), (1,)))
        else:
            p.gates.append(ir.Gate(['sx', 'rz', 'x'][r - 1], (int(q[0]),), (float(rng.uniform(-3, 3)),) if r == 2 else ()))
    p.measures.update({q: q for q in range(N)})
    m = Model()
    m.all(AD(2e-3, 0.1), ['sx', 'rz', 'x'])
    m.all(expand(AD(2e-3), AD(2e-3)), ['cx'])
    res = B200Simulator(precision='single', seed=5, noise_model=m.nm).run(p, shots=shots).result()
    assert res.metadata()['path'] == 'noisy_trajectories_kraus'
    assert_law(res.get_counts(), key_law(p, m), shots, 'long')


@gpu
@pytest.mark.parametrize('precision,N', [('single', 11), ('single', 12), ('single', 13), ('double', 11), ('double', 12),
                                         ('double', 13)])
def test_cta_branch_per_qubit_marginals_under_kraus_errors(precision, N):
    """Above 10 qubits a CTA runs one trajectory and reduces the stage qubit over its 8 warps.  One-qubit gates with
    one-qubit errors keep the state a product: each qubit's marginal is its own 1-qubit law."""
    shots = 1 << 17
    rng = np.random.RandomState(100 + N)
    p = ir.Program(N, N)
    for q in range(N):
        for _ in range(3):
            p.gates.append(ir.Gate('ry', (q,), (float(rng.uniform(0, np.pi)),)))
            name = ['sx', 'x', 'h', 'rz'][rng.randint(4)]
            p.gates.append(ir.Gate(name, (q,), (0.4,) if name == 'rz' else ()))
        p.measures[q] = q
    m = Model()
    m.all(AD(0.25, 0.1), ['sx'])
    m.all(compose(PD(0.3), CU(rx(0.5))), ['h'])
    m.all(TR(30e-6, 50e-6, 9e-6, 0.05), ['ry'])
    m.all(compose(DEP(0.1, 1), KR(user_gad_ops(0.3, 0.4))), ['x'])
    m.local(TR(10e-6, 8e-6, 20e-6), ['ry'], [N - 1])
    for q in range(0, N, 2):
        m.nm.add_readout_error(ReadoutError([[0.93, 0.07], [0.12, 0.88]]), [q])
    res = B200Simulator(precision=precision, seed=N, noise_model=m.nm).run(p, shots=shots).result()
    assert res.metadata()['path'] == 'noisy_trajectories_kraus'
    obs = np.zeros(N)
    for k, c in res.get_counts().items():
        bits = int(k, 2)
        for q in range(N):
            obs[q] += c * ((bits >> q) & 1)
    for q in range(N):
        sub = ir.Program(1, 1, gates=[ir.Gate(g.name, (0,), g.params) for g in p.gates if g.qubits == (q,)],
                         measures={0: 0})
        sm = Model()
        for name in ('sx', 'h', 'ry', 'x'):
            e = m.nm.gate_error(name, (q,))
            if e is not None:
                sm.all((e, m.supers[id(e)]), [name])
        if m.nm.readout_error(q) is not None:
            sm.nm.add_all_qubit_readout_error(m.nm.readout_error(q))
        law = key_law(sub, sm)
        assert abs(obs[q] / shots - law[1]) < weissman_tv_bound(2, shots, 1e-6 / N), (q, obs[q] / shots, law[1])


@gpu
@pytest.mark.parametrize('precision', ['double', 'single'])
def test_kraus_runs_are_reproducible_split_invariant_and_routed_per_circuit(precision):
    rng = np.random.RandomState(12)
    m = Model()
    m.all(DEP(0.05, 1), ['y'])
    m.all(PAULI([('Z', 0.1), ('I', 0.9)]), ['z'])
    m.all(compose(DEP(0.02, 1), TR(40e-6, 30e-6, 3e-6)), ['sx', 'x'])
    m.all(expand(AD(0.1), PD(0.2)), ['cx'])
    m.nm.add_all_qubit_readout_error(ReadoutError([[0.97, 0.03], [0.05, 0.95]]))

    def prog(N, names, n_gates):
        p = ir.Program(N, N, measures={q: q for q in range(N)})
        for _ in range(n_gates):
            q = rng.permutation(N)
            name = names[rng.randint(len(names))]
            p.gates.append(ir.Gate(name, (int(q[0]), int(q[1])), (), (1,)) if name in ('cz', 'cx') else ir.Gate(name, (int(q[0]),)))
        return p

    circs = [prog(3, ['h', 'y', 'z', 'cz'], 20), prog(4, ['h', 'sx', 'x', 'cx', 'y'], 30), prog(4, ['h', 'cz'], 10),
             prog(11, ['h', 'sx', 'cx', 'z'], 40), prog(5, ['h', 'y', 'cz'], 15)]
    paths = ['noisy_trajectories', 'noisy_trajectories_kraus', 'batch_small', 'noisy_trajectories_kraus',
             'noisy_trajectories']
    sim = B200Simulator(precision=precision, seed=321, noise_model=m.nm)
    res = sim.run(circs, shots=3000).result()
    assert [res.metadata(i)['path'] for i in range(len(circs))] == paths
    a = res.get_counts()
    assert sim.run(circs, shots=3000).result().get_counts() == a
    b = sim.run(circs[:2], shots=3000, stream_ids=[0, 1]).result().get_counts() + \
        sim.run(circs[2:], shots=3000, stream_ids=[2, 3, 4]).result().get_counts()
    assert a == b
    c = sim.run(circs, shots=3000, seed=322).result().get_counts()
    assert c[1] != a[1] and c[3] != a[3]
    # the Pauli-only circuits give what a model without the Kraus errors gives: their route did not change
    pauli_only = NoiseModel()
    pauli_only.add_all_qubit_quantum_error(m.nm.gate_error('y', (0,)), ['y'])
    pauli_only.add_all_qubit_quantum_error(m.nm.gate_error('z', (0,)), ['z'])
    pauli_only.add_all_qubit_readout_error(m.nm.readout_error(0))
    d = B200Simulator(precision=precision, seed=321, noise_model=pauli_only).run(
        [circs[0], circs[4]], shots=3000, stream_ids=[0, 4]).result().get_counts()
    assert d == [a[0], a[4]]


@gpu
def test_reference_flow_under_a_hardware_like_model(models):
    """The 70 transpiled fixtures of scale 0.25 in one run() call under tools/noise_bench.py's hardware-like model:
    depolarizing composed with thermal relaxation after sx / x / id, with two relaxations expanded after cx."""
    shots = 1 << 17
    T = [transpiled_fixture(models, '0.25', j, i) for j in range(7) for i in range(10)]
    m = hardware_model()
    res = B200Simulator(seed=2026, noise_model=m.nm).run(T, shots=shots).result()
    counts = res.get_counts()
    assert len(counts) == 70
    checked = 0
    for i, t in enumerate(T):
        assert sum(counts[i].values()) == shots
        assert res.metadata(i)['path'] == 'noisy_trajectories_kraus'
        p = ir.lower(t)
        device = None if p.n_qubits <= dm.MAX_QUBITS else 'cuda'        # graph 3: 10 qubits, the torch backend
        law = key_law(ir.Program(p.n_qubits, p.n_clbits, gates=list(p.gates), measures=dict(p.measures)), m, device)
        assert_law(counts[i], law, shots, i, alpha=1e-6 / 70)
        checked += 1
    assert checked == 70
