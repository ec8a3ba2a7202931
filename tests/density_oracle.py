"""Density-matrix law of a lowered program under a qcmrf_b200.noise.NoiseModel (test infrastructure).

A complex128 executor: after each ir.Gate the state becomes U rho U^dagger and then, when the model attaches a Pauli
error to the gate, sum_P p_P P rho P.  It reads the ir.Gate objects and the model's own entries (labels in Qiskit's
order) -- never the arrays noise.encode() hands the engine -- so that an encoding bug cannot hide in both.  key_law()
gives the distribution of the classical register with the per-clbit assignment matrices of the readout errors applied.

Two array backends run the same contractions: numpy (the default, up to MAX_QUBITS) and torch complex128 on a given
device (`device=`, up to MAX_QUBITS_TORCH, the engine's noisy limit).  A 13-qubit rho is 1 GiB and a 2-qubit
superoperator touches all of it once per gate, so at that size the law runs on the GPU.
"""
import numpy as np

MAX_QUBITS = 8
MAX_QUBITS_TORCH = 13                                            # kSmallMaxQubits
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


def initial_state(N, device=None):
    """|0...0><0...0| as a (2,) * 2N tensor: numpy when device is None, else torch complex128 on `device`."""
    if N > (MAX_QUBITS if device is None else MAX_QUBITS_TORCH):
        raise ValueError('density oracle: at most %d qubits on the %s backend'
                         % ((MAX_QUBITS, 'numpy') if device is None else (MAX_QUBITS_TORCH, 'torch')))
    if device is None:
        rho = np.zeros((1 << N, 1 << N), dtype=np.complex128)
    else:
        import torch
        rho = torch.zeros((1 << N, 1 << N), dtype=torch.complex128, device=device)
    rho[0, 0] = 1.0
    return rho.reshape((2,) * (2 * N))


def operator(S, T):
    """S (a numpy operator, or one already in T's backend) in T's backend."""
    if isinstance(T, np.ndarray) or not isinstance(S, np.ndarray):
        return S
    import torch
    return torch.tensor(np.asarray(S, dtype=np.complex128), device=T.device)      # a copy: S may be read-only


def _apply(T, S, axes):
    """Contract the operator S (on len(axes) bits, most significant first) into the tensor axes `axes`."""
    m = len(axes)
    if isinstance(T, np.ndarray):
        out = np.tensordot(S.reshape((2,) * (2 * m)), T, axes=(list(range(m, 2 * m)), axes))
        return np.moveaxis(out, list(range(m)), axes)
    import torch
    out = torch.tensordot(operator(S, T).reshape((2,) * (2 * m)), T, dims=(list(range(m, 2 * m)), list(axes)))
    return torch.movedim(out, list(range(m)), list(axes))


def apply_controlled(T, g, N):
    """U rho U^dagger for a gate g of 3 or more qubits (no error): its base 2x2 on the target's row axis where every
    control's row axis holds its value, then the conjugate on the column axes likewise.  Exact, and without the
    2^k x 2^k matrix, which at 13 qubits would be 1 GiB per gate."""
    B = g.base_matrix()
    for off, op in ((0, B), (N, B.conj())):
        axis = lambda q: off + N - 1 - q                         # row axis of bit q: N-1-q, column axis: 2N-1-q
        idx = [slice(None)] * (2 * N)
        for q, v in zip(g.controls, g.ctrl_values):
            idx[axis(q)] = int(v)
        t = axis(g.target) - sum(axis(q) < axis(g.target) for q in g.controls)   # in the slice, whose control axes are gone
        sub = T[tuple(idx)]
        T[tuple(idx)] = _apply(sub, op, [t])
    return T


def run(prog, model=None, device=None):
    """rho (2^N x 2^N complex128) after the program's gates from |0...0><0...0|: a numpy array, or a torch tensor
    on `device`."""
    N = prog.n_qubits
    T = initial_state(N, device)
    supers = {}                                                  # superoperator per (gate, error): fixtures repeat them
    for g in prog.gates:
        err = _gate_error(model, g)
        rows = [N - 1 - q for q in reversed(g.qubits)]           # tensor axis of row bit q: N-1-q
        cols = [2 * N - 1 - q for q in reversed(g.qubits)]       # of column bit q: 2N-1-q
        if len(g.qubits) > 2:
            if err is not None:
                raise ValueError('error on a gate of %d qubits' % len(g.qubits))
            T = apply_controlled(T, g, N)                        # U rho U^dagger
            continue
        key = (g.name, g.params, g.ctrl_values, len(g.qubits), id(err))
        S = supers.get(key)
        if S is None:
            U = g.matrix()
            terms = [(1.0, U)] if err is None else [(p, _label_matrix(label) @ U) for label, p in err.to_labels()]
            S = supers[key] = operator(sum(p * np.kron(A, A.conj()) for p, A in terms), T)
        T = _apply(T, S, rows + cols)                            # one superoperator on (rows, columns)
    return T.reshape(1 << N, 1 << N)


def diagonal(rho):
    """Real part of rho's diagonal as a numpy float64 vector, from either backend (a vector is taken as the
    diagonal itself)."""
    if isinstance(rho, np.ndarray):
        return np.real(rho if rho.ndim == 1 else np.diag(rho))
    return rho.diagonal().real.cpu().numpy()


def key_law(prog, model=None, rho=None, device=None):
    """Distribution over classical-register integers (clbit c = bit c): outcomes from diag(rho), keys from the
    program's measurements (unmeasured clbits 0), each measured clbit then read through its qubit's readout error.
    `rho` may be given as its diagonal alone."""
    if rho is None:
        rho = run(prog, model, device)
    N, ncl = prog.n_qubits, max(prog.n_clbits, 1)
    p = np.clip(diagonal(rho), 0.0, None)
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
