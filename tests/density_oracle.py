"""Density-matrix law of a lowered program under a qcmrf_b200.noise.NoiseModel (test infrastructure).

A complex128 executor for programs of up to 8 qubits: after each ir.Gate the state becomes U rho U^dagger and then,
when the model attaches a Pauli error to the gate, sum_P p_P P rho P.  It reads the ir.Gate objects and the model's
own entries (labels in Qiskit's order) -- never the arrays noise.encode() hands the engine -- so that an encoding
bug cannot hide in both.  key_law() gives the distribution of the classical register with the per-clbit
assignment matrices of the readout errors applied.
"""
import numpy as np

MAX_QUBITS = 8
_PAULI = {'I': np.eye(2, dtype=np.complex128), 'X': np.array([[0, 1], [1, 0]], dtype=np.complex128),
          'Y': np.array([[0, -1j], [1j, 0]], dtype=np.complex128), 'Z': np.diag([1.0, -1.0]).astype(np.complex128)}


def _gate_error(model, gate):
    """The model's error after `gate`: a qubit-specific entry wins over the all-qubit one."""
    if model is None:
        return None
    e = model._local_gate.get((gate.name, tuple(gate.qubits)))
    return e if e is not None else model._all_gate.get(gate.name)


def _readout_error(model, qubit):
    if model is None:
        return None
    e = model._local_readout.get(qubit)
    return e if e is not None else model._all_readout


def _label_matrix(label):
    """Pauli string -> matrix on the gate's qubits, index bit j <-> qubits[j] (the last character acts on qubits[0])."""
    m = np.ones((1, 1), dtype=np.complex128)
    for ch in label:
        m = np.kron(m, _PAULI[ch])
    return m


def _apply(T, S, axes):
    """Contract the operator S (on len(axes) bits, most significant first) into the tensor axes `axes`."""
    m = len(axes)
    out = np.tensordot(S.reshape((2,) * (2 * m)), T, axes=(list(range(m, 2 * m)), axes))
    return np.moveaxis(out, list(range(m)), axes)


def run(prog, model=None):
    """rho (2^N x 2^N complex128) after the program's gates from |0...0><0...0|."""
    N = prog.n_qubits
    if N > MAX_QUBITS:
        raise ValueError('density oracle: at most %d qubits' % MAX_QUBITS)
    rho = np.zeros((1 << N, 1 << N), dtype=np.complex128)
    rho[0, 0] = 1.0
    T = rho.reshape((2,) * (2 * N))
    supers = {}                                                  # superoperator per (gate, error): fixtures repeat them
    for g in prog.gates:
        err = _gate_error(model, g)
        rows = [N - 1 - q for q in reversed(g.qubits)]           # tensor axis of row bit q: N-1-q
        cols = [2 * N - 1 - q for q in reversed(g.qubits)]       # of column bit q: 2N-1-q
        if len(g.qubits) > 2:
            if err is not None:
                raise ValueError('error on a gate of %d qubits' % len(g.qubits))
            U = g.matrix()                                       # U rho U^dagger
            T = _apply(_apply(T, U, rows), U.conj(), cols)
            continue
        key = (g.name, g.params, g.ctrl_values, len(g.qubits), id(err))
        S = supers.get(key)
        if S is None:
            U = g.matrix()
            terms = [(1.0, U)] if err is None else [(p, _label_matrix(label) @ U) for label, p in err.to_labels()]
            S = supers[key] = sum(p * np.kron(A, A.conj()) for p, A in terms)
        T = _apply(T, S, rows + cols)                            # one superoperator on (rows, columns)
    return T.reshape(1 << N, 1 << N)


def key_law(prog, model=None, rho=None):
    """Distribution over classical-register integers (clbit c = bit c): outcomes from diag(rho), keys from the
    program's measurements (unmeasured clbits 0), each measured clbit then read through its qubit's readout error."""
    if rho is None:
        rho = run(prog, model)
    N, ncl = prog.n_qubits, max(prog.n_clbits, 1)
    p = np.clip(np.real(np.diag(rho)), 0.0, None)
    idx = np.arange(1 << N)
    key = np.zeros(1 << N, dtype=np.int64)
    for c, q in prog.measures.items():
        key |= ((idx >> q) & 1) << c
    law = np.zeros(1 << ncl)
    np.add.at(law, key, p)
    L = law.reshape((2,) * ncl)
    for c, q in sorted(prog.measures.items()):
        e = _readout_error(model, q)
        if e is None:
            continue
        ax = ncl - 1 - c
        L = np.moveaxis(np.tensordot(L, e.probabilities, axes=([ax], [0])), -1, ax)
    return L.reshape(-1)
