"""Gate errors and readout errors for noisy shot simulation (Aer's names and conventions).

    from qcmrf_b200.noise import NoiseModel, depolarizing_error, thermal_relaxation_error, ReadoutError
    nm = NoiseModel()
    t1q = thermal_relaxation_error(100e-6, 80e-6, 35.5e-9)
    t2q = thermal_relaxation_error(100e-6, 80e-6, 300e-9)
    nm.add_all_qubit_quantum_error(depolarizing_error(1e-3, 1).compose(t1q), ['sx', 'x', 'id'])
    nm.add_all_qubit_quantum_error(depolarizing_error(1e-2, 2).compose(t2q.expand(t2q)), ['cx'])
    nm.add_all_qubit_readout_error(ReadoutError([[0.98, 0.02], [0.02, 0.98]]))
    counts = B200Simulator(noise_model=nm).run(circuits, shots=10000).result().get_counts()

Semantics (as Aer): every gate is applied and then its error channel acts on the gate's qubits; measurements are
deferred to the end of the program; each measured clbit is flipped by its measured qubit's readout error.  Every
shot is an independent trajectory with its own error draws, outcome and readout draws, so the counts are i.i.d.
samples of the density-matrix law.

An error (QuantumError) is an ordered list of at most MAX_STAGES stages on its 1 or 2 qubits, each a Pauli channel
or a 1-qubit channel in canonical Kraus form (at most 4 operators).  A trajectory unravels a Kraus stage by choosing
operator K_i with probability tr(K_i^dagger K_i rho_q) on its current state and renormalising, which has the
stage's density-matrix law.

Errors attach to the primitive gates the circuit lowers to (qcmrf_b200.ir): a ``swap`` is three ``cx`` and a
composite instruction is its definition's gates, so errors are given for primitive gate names only.
"""
import numpy as np

from . import ir

__all__ = ['QuantumError', 'PauliError', 'pauli_error', 'depolarizing_error', 'amplitude_damping_error',
           'phase_damping_error', 'phase_amplitude_damping_error', 'thermal_relaxation_error', 'kraus_error',
           'coherent_unitary_error', 'ReadoutError', 'NoiseModel']

_PAULI_CODE = {'I': 0, 'X': 1, 'Y': 2, 'Z': 3}
#: gate names lowering keeps as primitives, with their qubit count (None: any, the multi-controlled gates)
_ARITY = dict([(n, 1) for n in list(ir._ONEQ) + list(ir._PARAM1Q) + ['u']] +
              [(n, 2) for n in ir._CTRL_BASE if n not in ('mcx', 'mcp')] + [('mcx', None), ('mcp', None)])
#: most Pauli terms of one channel (a 2-qubit error)
MAX_PAULIS = 16
#: most stages of one error, and most operators of one Kraus stage (every 1-qubit channel has Choi rank <= 4)
MAX_STAGES = 4
MAX_KRAUS = 4
#: tolerance of sum_i K_i^dagger K_i = I (user-computed products such as sqrt(1-a) sqrt(1-p1) carry rounding)
KRAUS_ATOL = 1e-10


def _choi(S):
    """Choi matrix of a 1-qubit superoperator S (acting on row-major vec(rho), S = sum K (x) conj(K)), and back:
    the same index shuffle (a, b, c, d) -> (a, c, b, d) both ways."""
    return S.reshape(2, 2, 2, 2).transpose(0, 2, 1, 3).reshape(4, 4)


def _superop(ops):
    return sum(np.kron(K, K.conj()) for K in ops)


def _check_tp(ops, what):
    dev = np.abs(sum(K.conj().T @ K for K in ops) - np.eye(ops[0].shape[0])).max()
    if not dev <= KRAUS_ATOL:
        raise ValueError('%s: sum of K^dagger K differs from the identity by %.3g (more than %g)' % (what, dev, KRAUS_ATOL))


def _canonical_kraus(S, what):
    """Canonical Kraus operators (n, 2, 2) of the 1-qubit channel with superoperator S: the eigenvectors of its Choi
    matrix with eigenvalues above 1e-15 of its trace, scaled by their square roots."""
    J = _choi(S)
    J = 0.5 * (J + J.conj().T)
    lam, V = np.linalg.eigh(J)
    keep = np.nonzero(lam > 1e-15 * np.real(np.trace(J)))[0][::-1]
    ops = np.array([np.sqrt(lam[k]) * V[:, k].reshape(2, 2) for k in keep], dtype=np.complex128)
    if not 1 <= len(ops) <= MAX_KRAUS:
        raise ValueError('%s: the channel has %d canonical Kraus operators' % (what, len(ops)))
    _check_tp(ops, what)
    ops.setflags(write=False)
    return ops


class QuantumError:
    """A gate error: an ordered list of at most MAX_STAGES stages on the error's ``num_qubits`` (1 or 2) qubits.

    ``stages`` holds ``('pauli', probs, qubits)`` -- a Pauli channel (probabilities as PauliError.probs) on the
    error's qubits ``qubits`` (a tuple of 1 or 2 positions) -- and ``('kraus', ops, qubit)`` -- the 1-qubit channel
    rho -> sum_i K_i rho K_i^dagger with canonical Kraus operators ``ops`` (n <= 4, 2x2) on the error's qubit
    ``qubit``.  Stages apply in order.  Position j is the gate's j-th qubit (for ``cx``, 0 is the control)."""

    def __init__(self, num_qubits, stages):
        self.num_qubits = int(num_qubits)
        self.stages = tuple(stages)
        if self.num_qubits > 2:
            raise ValueError('errors act on 1 or 2 qubits, not %d' % self.num_qubits)
        if len(self.stages) > MAX_STAGES:
            raise ValueError('an error holds at most %d stages, not %d' % (MAX_STAGES, len(self.stages)))

    @staticmethod
    def _stage_ideal(st):
        if st[0] == 'pauli':
            return not (st[1][1:] > 0).any()
        return np.abs(_superop(st[1]) - np.eye(4)).max() <= 1e-14

    def ideal(self):
        """True when every stage is the identity channel (a Kraus stage within 1e-14 of it as a superoperator)."""
        return all(self._stage_ideal(st) for st in self.stages)

    def is_single_pauli(self):
        """True for one Pauli stage on all the error's qubits: the case qcm_run_noisy_small runs."""
        return len(self.stages) == 1 and self.stages[0][0] == 'pauli' and len(self.stages[0][2]) == self.num_qubits

    def compose(self, other):
        """This error, then `other` (on the same qubits)."""
        other = _as_error(other)
        if other.num_qubits != self.num_qubits:
            raise ValueError('compose: a %d-qubit error and a %d-qubit error' % (self.num_qubits, other.num_qubits))
        return QuantumError(self.num_qubits, self.stages + other.stages)

    def tensor(self, other):
        """The 2-qubit error with `other` on qubit 0 and this error on qubit 1 (Aer's order)."""
        return _product(_as_error(other), self)

    def expand(self, other):
        """The 2-qubit error with this error on qubit 0 and `other` on qubit 1 (Aer's order)."""
        return _product(self, _as_error(other))

    def __repr__(self):
        return 'QuantumError(%d qubits, %s)' % (self.num_qubits, ', '.join(
            '%s on %s' % (st[0], st[2]) for st in self.stages))


def _as_error(e):
    if not isinstance(e, QuantumError):
        raise ValueError('not a QuantumError: %r' % (e,))
    return e


def _shift(st, by):
    if st[0] == 'pauli':
        return ('pauli', st[1], tuple(q + by for q in st[2]))
    return ('kraus', st[1], st[2] + by)


def _product(q0, q1):
    """q0 on qubit 0, q1 on qubit 1."""
    if q0.num_qubits != 1 or q1.num_qubits != 1:
        raise ValueError('tensor / expand: only 1-qubit errors combine (the result would have %d qubits; at most 2 '
                         'are supported)' % (q0.num_qubits + q1.num_qubits))
    return QuantumError(2, q0.stages + tuple(_shift(st, 1) for st in q1.stages))


class PauliError(QuantumError):
    """A Pauli channel on 1 or 2 qubits: rho -> sum_k p_k P_k rho P_k.

    ``probs[k]`` is the probability of the Pauli whose code on the channel's qubit j is ``(k >> 2j) & 3``
    (0 = I, 1 = X, 2 = Y, 3 = Z); k = 0 is the identity."""

    def __init__(self, n_qubits, probs):
        probs = np.asarray(probs, dtype=np.float64)
        probs.setflags(write=False)
        super().__init__(n_qubits, [('pauli', probs, tuple(range(int(n_qubits))))])
        self.probs = probs

    def ideal(self):
        """True when the channel never applies a non-identity Pauli."""
        return not (self.probs[1:] > 0).any()

    def to_labels(self):
        """[(label, p)] with Qiskit's order (the last character acts on the first qubit), p > 0 only."""
        out = []
        for k, p in enumerate(self.probs):
            if p > 0:
                out.append((''.join('IXYZ'[(k >> (2 * j)) & 3] for j in reversed(range(self.num_qubits))), float(p)))
        return out

    def __repr__(self):
        return 'PauliError(%r)' % (self.to_labels(),)


def pauli_error(noise_ops):
    """Pauli channel from [(label, p), ...]: labels of 1 or 2 characters over IXYZ, all of one length; the last
    character acts on the gate's first qubit (for ``cx``, the control).  p >= 0, summing to 1 within 1e-12;
    a label may repeat (its probabilities add)."""
    ops = list(noise_ops)
    if not ops:
        raise ValueError('pauli_error: no Pauli terms')
    n = None
    probs = None
    for item in ops:
        try:
            label, p = item
        except (TypeError, ValueError):
            raise ValueError('pauli_error: terms are (label, probability) pairs, got %r' % (item,))
        if not isinstance(label, str) or not 1 <= len(label) <= 2 or any(ch not in _PAULI_CODE for ch in label):
            raise ValueError('pauli_error: label %r is not 1 or 2 characters over IXYZ' % (label,))
        if n is None:
            n = len(label)
            probs = np.zeros(4 ** n)
        elif len(label) != n:
            raise ValueError('pauli_error: labels of different lengths')
        p = float(p)
        if not np.isfinite(p) or p < 0:
            raise ValueError('pauli_error: probability %r of %r is not >= 0' % (p, label))
        k = 0
        for j, ch in enumerate(reversed(label)):
            k |= _PAULI_CODE[ch] << (2 * j)
        probs[k] += p
    if abs(probs.sum() - 1.0) > 1e-12:
        raise ValueError('pauli_error: probabilities sum to %.17g, not 1' % probs.sum())
    return PauliError(n, probs)


def depolarizing_error(param, num_qubits):
    """Aer's depolarizing channel (1 - lam) rho + lam I / 2^n for n in {1, 2}, 0 <= lam <= 4^n / (4^n - 1): the
    identity with probability 1 - lam (4^n - 1) / 4^n, each other Pauli with lam / 4^n."""
    n = int(num_qubits)
    if n not in (1, 2) or n != num_qubits:
        raise ValueError('depolarizing_error: num_qubits must be 1 or 2')
    lam = float(param)
    d2 = 4 ** n
    if not np.isfinite(lam) or lam < 0 or lam > d2 / (d2 - 1):
        raise ValueError('depolarizing_error: lambda %r outside [0, %g]' % (param, d2 / (d2 - 1)))
    probs = np.full(d2, lam / d2)
    probs[0] = 1.0 - lam * (d2 - 1) / d2
    return PauliError(n, probs)


def _param(x, what):
    x = float(x)
    if not np.isfinite(x):
        raise ValueError('%s: %r is not finite' % (what, x))
    return x


def _damping(a, p1, c, what):
    """QuantumError of the 1-qubit channel rho_11 -> (1 - a) rho_11 + a p1 tr(rho), rho_01 -> c rho_01 (c real)."""
    S = np.zeros((4, 4))
    S[0, 0], S[0, 3] = 1 - a * p1, a * (1 - p1)           # vec(rho) = (rho_00, rho_01, rho_10, rho_11)
    S[3, 0], S[3, 3] = a * p1, 1 - a + a * p1
    S[1, 1] = S[2, 2] = c
    return QuantumError(1, [('kraus', _canonical_kraus(S.astype(np.complex128), what), 0)])


def _check_population(p1, what):
    p1 = _param(p1, what)
    if not 0 <= p1 <= 1:
        raise ValueError('%s: excited_state_population %r outside [0, 1]' % (what, p1))
    return p1


def amplitude_damping_error(param_amp, excited_state_population=0):
    """Generalised amplitude damping: rho_11 -> (1 - a) rho_11 + a p1, rho_01 -> sqrt(1 - a) rho_01."""
    a = _param(param_amp, 'amplitude_damping_error')
    p1 = _check_population(excited_state_population, 'amplitude_damping_error')
    if not 0 <= a <= 1:
        raise ValueError('amplitude_damping_error: param_amp %r outside [0, 1]' % a)
    return _damping(a, p1, np.sqrt(1 - a), 'amplitude_damping_error')


def phase_damping_error(param_phase):
    """Phase damping: the diagonal is kept, rho_01 -> sqrt(1 - b) rho_01."""
    b = _param(param_phase, 'phase_damping_error')
    if not 0 <= b <= 1:
        raise ValueError('phase_damping_error: param_phase %r outside [0, 1]' % b)
    return _damping(0.0, 0.0, np.sqrt(1 - b), 'phase_damping_error')


def phase_amplitude_damping_error(param_amp, param_phase, excited_state_population=0):
    """rho_11 -> (1 - a) rho_11 + a p1, rho_01 -> sqrt(1 - a - b) rho_01; a, b >= 0, a + b <= 1."""
    what = 'phase_amplitude_damping_error'
    a, b = _param(param_amp, what), _param(param_phase, what)
    p1 = _check_population(excited_state_population, what)
    if a < 0 or b < 0 or a + b > 1:
        raise ValueError('%s: param_amp %r and param_phase %r must be >= 0 with a sum <= 1' % (what, a, b))
    return _damping(a, p1, np.sqrt(1 - a - b), what)


def thermal_relaxation_error(t1, t2, time, excited_state_population=0):
    """Thermal relaxation for `time`: rho_11 -> p1 + (rho_11 - p1) e^(-time/t1), rho_01 -> rho_01 e^(-time/t2).
    t1, t2 > 0 (either may be inf), t2 <= 2 t1, time >= 0.  Aer writes T2 <= T1 as a mixture with resets; this is
    the same channel in Kraus form."""
    what = 'thermal_relaxation_error'
    t1, t2, time = float(t1), float(t2), _param(time, what)
    p1 = _check_population(excited_state_population, what)
    if not t1 > 0 or not t2 > 0 or np.isnan(t1) or np.isnan(t2):
        raise ValueError('%s: t1 %r and t2 %r must be > 0' % (what, t1, t2))
    if t2 > 2 * t1:
        raise ValueError('%s: t2 %r above 2 t1 (%r) is not a physical channel' % (what, t2, 2 * t1))
    if time < 0:
        raise ValueError('%s: time %r < 0' % (what, time))
    return _damping(-np.expm1(-time / t1), p1, np.exp(-time / t2), what)


def kraus_error(noise_ops):
    """The channel rho -> sum_i K_i rho K_i^dagger.  1-qubit operators (2x2), or 2-qubit ones (4x4) whose channel is a
    tensor product of two 1-qubit channels; sum_i K_i^dagger K_i = I within 1e-10."""
    try:
        ops = np.array([np.asarray(K, dtype=np.complex128) for K in noise_ops])
    except (TypeError, ValueError):
        raise ValueError('kraus_error: operators of one square shape are needed')
    if ops.ndim != 3 or not len(ops) or ops.shape[1:] not in ((2, 2), (4, 4)):
        raise ValueError('kraus_error: operators must all be 2x2 (or 4x4 for a product of two 1-qubit channels), '
                         'got shape %r' % (ops.shape,))
    if not np.isfinite(ops).all():
        raise ValueError('kraus_error: operators must be finite')
    _check_tp(ops, 'kraus_error')
    if ops.shape[1] == 2:
        return QuantumError(1, [('kraus', _canonical_kraus(_superop(ops), 'kraus_error'), 0)])
    # 2 qubits (index bit j <-> error qubit j).  The Choi matrix of a product channel is the product of the 1-qubit
    # ones, which are its partial traces over the other qubit / 2.
    T = sum(np.outer(K.reshape(-1), K.conj().reshape(-1)) for K in ops).reshape((2,) * 8)
    # T axes: (out1, out0, in1, in0, out1', out0', in1', in0')
    J1 = np.einsum('axbycxdy->abcd', T) / 2
    J0 = np.einsum('xaybxcyd->abcd', T) / 2
    if np.abs(np.einsum('abcd,efgh->aebfcgdh', J1, J0) - T).max() > KRAUS_ATOL:
        raise ValueError('kraus_error: this 2-qubit channel is not a tensor product of 1-qubit channels; 2-qubit '
                         'Kraus errors are supported as tensor products of 1-qubit ones')
    e0 = QuantumError(1, [('kraus', _canonical_kraus(_choi(J0.reshape(4, 4)), 'kraus_error'), 0)])
    e1 = QuantumError(1, [('kraus', _canonical_kraus(_choi(J1.reshape(4, 4)), 'kraus_error'), 0)])
    return e0.expand(e1)


def coherent_unitary_error(unitary):
    """The unitary channel rho -> U rho U^dagger of a 2x2 unitary (within 1e-10)."""
    U = np.asarray(unitary, dtype=np.complex128)
    if U.shape != (2, 2) or not np.isfinite(U).all() or np.abs(U.conj().T @ U - np.eye(2)).max() > KRAUS_ATOL:
        raise ValueError('coherent_unitary_error: a 2x2 unitary is needed')
    ops = U.reshape(1, 2, 2).copy()
    ops.setflags(write=False)
    return QuantumError(1, [('kraus', ops, 0)])


class ReadoutError:
    """Classical assignment error of one measured qubit: ``probabilities[v][r]`` = P(read r | outcome v),
    i.e. [[P(0|0), P(1|0)], [P(0|1), P(1|1)]]; each row sums to 1 within 1e-12."""

    def __init__(self, probabilities):
        a = np.array(probabilities, dtype=np.float64)
        if a.shape != (2, 2):
            raise ValueError('ReadoutError: a 2x2 matrix of probabilities is needed (one qubit)')
        if not np.isfinite(a).all() or (a < 0).any() or (np.abs(a.sum(axis=1) - 1.0) > 1e-12).any():
            raise ValueError('ReadoutError: each row must hold probabilities >= 0 that sum to 1')
        a.setflags(write=False)
        self.probabilities = a

    def ideal(self):
        return self.probabilities[0, 1] == 0 and self.probabilities[1, 0] == 0

    def __repr__(self):
        return 'ReadoutError(%r)' % (self.probabilities.tolist(),)


def _gate_names(instructions):
    if isinstance(instructions, str):
        instructions = [instructions]
    out = []
    for name in instructions:
        if not isinstance(name, str):
            raise ValueError('gate names are strings, got %r' % (name,))
        canon = ir._ALIASES.get(name.lower(), name.lower())
        if canon not in _ARITY:
            raise ValueError('no error can attach to %r: it is not a primitive gate of the lowered program (swap is '
                             'three cx, measure is deferred, composite instructions lower to their gates)' % name)
        out.append(canon)
    if not out:
        raise ValueError('no gate names given')
    return out


def _check_error(error):
    if not isinstance(error, QuantumError):
        raise ValueError('a gate error is a QuantumError (pauli_error, depolarizing_error, thermal_relaxation_error, '
                         'kraus_error, ...), got %r' % (error,))


class NoiseModel:
    """Gate errors keyed by (gate name, qubits) and readout errors keyed by qubit.  A qubit-specific entry wins over
    the all-qubit one; a second error for the same key is refused (errors are not composed)."""

    def __init__(self):
        self._all_gate = {}          # name -> QuantumError
        self._local_gate = {}        # (name, qubits tuple) -> QuantumError
        self._all_readout = None
        self._local_readout = {}     # qubit -> ReadoutError

    def __repr__(self):
        return 'NoiseModel(gates=%s, readout=%s)' % (sorted(set(self._all_gate) | {k[0] for k in self._local_gate}),
                                                     'all' if self._all_readout is not None else sorted(self._local_readout))

    def is_ideal(self):
        """True when every error of the model is the identity channel."""
        return (all(e.ideal() for e in self._all_gate.values()) and all(e.ideal() for e in self._local_gate.values())
                and (self._all_readout is None or self._all_readout.ideal())
                and all(r.ideal() for r in self._local_readout.values()))

    def add_all_qubit_quantum_error(self, error, instructions):
        _check_error(error)
        names = _gate_names(instructions)
        for name in names:
            if _ARITY[name] is not None and _ARITY[name] != error.num_qubits:
                raise ValueError('a %d-qubit error cannot attach to %r, a %d-qubit gate' % (error.num_qubits, name, _ARITY[name]))
            if name in self._all_gate:
                raise ValueError('an all-qubit error for %r is already in the model (errors are not composed)' % name)
        for name in names:
            self._all_gate[name] = error

    def add_quantum_error(self, error, instructions, qubits):
        _check_error(error)
        names = _gate_names(instructions)
        qs = tuple(int(q) for q in qubits)
        if len(qs) != error.num_qubits or len(set(qs)) != len(qs) or min(qs) < 0:
            raise ValueError('qubits %r do not fit a %d-qubit error' % (tuple(qubits), error.num_qubits))
        for name in names:
            if _ARITY[name] is not None and _ARITY[name] != len(qs):
                raise ValueError('%r acts on %d qubits, not %d' % (name, _ARITY[name], len(qs)))
            if (name, qs) in self._local_gate:
                raise ValueError('an error for %r on qubits %r is already in the model (errors are not composed)' % (name, qs))
        for name in names:
            self._local_gate[(name, qs)] = error

    def add_all_qubit_readout_error(self, error):
        if not isinstance(error, ReadoutError):
            error = ReadoutError(error)
        if self._all_readout is not None:
            raise ValueError('an all-qubit readout error is already in the model')
        self._all_readout = error

    def add_readout_error(self, error, qubits):
        if not isinstance(error, ReadoutError):
            error = ReadoutError(error)
        qs = [int(q) for q in qubits]
        if len(qs) != 1 or qs[0] < 0:
            raise ValueError('a readout error acts on one qubit')
        if qs[0] in self._local_readout:
            raise ValueError('a readout error for qubit %d is already in the model' % qs[0])
        self._local_readout[qs[0]] = error

    # -- lookups ---------------------------------------------------------------------------------
    def gate_error(self, name, qubits):
        """The QuantumError that follows gate `name` on `qubits` (controls..., target), or None."""
        e = self._local_gate.get((name, tuple(qubits)))
        return e if e is not None else self._all_gate.get(name)

    def readout_error(self, qubit):
        e = self._local_readout.get(int(qubit))
        return e if e is not None else self._all_readout

    def readout_table(self, prog):
        """(64, 2) flip probabilities per clbit of `prog`: P(read 1 | 0), P(read 0 | 1) of its measured qubit's readout
        error; zero for unmeasured clbits and qubits without one."""
        t = np.zeros((64, 2))
        for c, q in prog.measures.items():
            e = self.readout_error(q)
            if e is not None:
                t[c] = e.probabilities[0, 1], e.probabilities[1, 0]
        return t


class EncodedNoise:
    """A lowered program encoded for the trajectory kernel (see encode()).  One record per gate: target, control mask,
    control-value mask (uint64 here, uint32 in the engine's qcm_gate: noisy circuits have at most 13 qubits), the
    2x2 matrix (fp64, row-major re/im) and an error index (-1: no error).

    One error record per distinct (error, gate qubits): ``err_n_stages`` stages, stage j a Pauli channel
    (``err_kind`` 0, ``err_index`` into the channel records) or a 1-qubit Kraus channel (kind 1, index into the
    Kraus records).  Channel records: cumulative Pauli probabilities and their physical qubits.  Kraus records: up
    to 4 operators (fp64, row-major re/im), their count and their physical qubit.

    ``kraus`` says which entry point runs the circuit.  False when every error that applies is one Pauli stage:
    then error k IS channel k (``channel`` indexes both) and qcm_run_noisy_small runs it; True otherwise
    (qcm_run_noisy_small_kraus)."""
    __slots__ = ('n_qubits', 'n_gates', 'target', 'ctrl_mask', 'ctrl_value', 'matrix', 'channel', 'cum', 'n_paulis',
                 'chan_qubits', 'err_n_stages', 'err_kind', 'err_index', 'kraus_ops', 'kraus_n_ops', 'kraus_qubit',
                 'kraus', 'clbit_map', 'readout', 'gate_noisy', 'readout_noisy', 'n_clbits')

    @property
    def noisy(self):
        return self.gate_noisy or self.readout_noisy


class _Records:
    def __init__(self):
        self.index = {}
        self.cum, self.n, self.qubits = [], [], []                       # Pauli channels
        self.kops, self.kn, self.kq = [], [], []                         # Kraus stages
        self.err_n, self.err_kind, self.err_index = [], [], []          # errors
        self.kraus = False

    def _channel(self, probs, qubits):
        c = np.zeros(MAX_PAULIS)
        c[:probs.size] = np.cumsum(probs)
        c[probs.size - 1:] = 1.0                      # the last entry catches every uniform in [0, 1)
        self.cum.append(c)
        self.n.append(probs.size)
        self.qubits.append((qubits[0], qubits[1] if len(qubits) > 1 else -1))
        return len(self.cum) - 1

    def _kraus(self, ops, qubit):
        k = np.zeros((MAX_KRAUS, 8))
        k[:len(ops), 0::2] = ops.reshape(-1, 4).real
        k[:len(ops), 1::2] = ops.reshape(-1, 4).imag
        self.kops.append(k)
        self.kn.append(len(ops))
        self.kq.append(qubit)
        return len(self.kops) - 1

    def get(self, err, qubits):
        """Error index of `err` on `qubits` (-1 for an error that never applies)."""
        if err is None or err.ideal():
            return -1
        if len(qubits) > 2:
            raise ValueError('an error is attached to a gate on %d qubits: transpile first' % len(qubits))
        if len(qubits) != err.num_qubits:
            raise ValueError('a %d-qubit error cannot follow a gate on qubits %r' % (err.num_qubits, tuple(qubits)))
        key = (id(err), tuple(qubits))
        k = self.index.get(key)
        if k is None:
            k = self.index[key] = len(self.err_n)
            kind, index = [0] * MAX_STAGES, [0] * MAX_STAGES
            for j, st in enumerate(err.stages):
                if st[0] == 'pauli':
                    kind[j], index[j] = 0, self._channel(st[1], [qubits[q] for q in st[2]])
                else:
                    kind[j], index[j] = 1, self._kraus(st[1], qubits[st[2]])
            self.err_n.append(len(err.stages))
            self.err_kind.append(kind)
            self.err_index.append(index)
            self.kraus |= not err.is_single_pauli()
        return k


def encode(prog, model):
    """Encode a lowered Program (an ir.BasisProgram straight from its arrays) with the errors `model` attaches to
    its gates.  Raises ValueError for an error on a gate of 3 or more qubits ("transpile first")."""
    N = prog.n_qubits
    ch = _Records()
    if isinstance(prog, ir.BasisProgram):
        bk, bq, bc = prog.bk.astype(np.int64), prog.bq.astype(np.int64), prog.bc.astype(np.int64)
        G = bk.size
        target = bq.astype(np.int32)
        ctrl = np.where(bk == 4, np.left_shift(np.uint64(1), np.maximum(bc, 0).astype(np.uint64)), np.uint64(0))
        cval = ctrl                                    # cx: control value 1
        mats = np.zeros((G, 2, 2), dtype=np.complex128)
        for k, name in enumerate(ir.BASIS_KINDS):
            sel = bk == k
            if not sel.any():
                continue
            if name == 'rz':
                h = 0.5 * prog.bp[sel]
                mats[sel, 0, 0], mats[sel, 1, 1] = np.exp(-1j * h), np.exp(1j * h)
            else:
                mats[sel] = ir.one_qubit_matrix('x' if name == 'cx' else name)
        channel = np.full(G, -1, dtype=np.int32)
        for k, name in enumerate(ir.BASIS_KINDS):            # one lookup per distinct (kind, qubits) of the program
            sel = np.nonzero(bk == k)[0]
            if not sel.size:
                continue
            keys = np.stack([bc[sel], bq[sel]], axis=1) if name == 'cx' else bq[sel, None]
            uniq, inv = np.unique(keys, axis=0, return_inverse=True)
            ids = np.array([ch.get(model.gate_error(name, tuple(int(q) for q in u)), tuple(int(q) for q in u))
                            for u in uniq], dtype=np.int32)
            channel[sel] = ids[inv.reshape(-1)]
    else:
        gates = prog.gates
        G = len(gates)
        target = np.empty(G, dtype=np.int32)
        ctrl = np.zeros(G, dtype=np.uint64)
        cval = np.zeros(G, dtype=np.uint64)
        mats = np.empty((G, 2, 2), dtype=np.complex128)
        channel = np.empty(G, dtype=np.int32)
        for i, g in enumerate(gates):
            target[i] = g.target
            m = v = 0
            for c, b in zip(g.controls, g.ctrl_values):
                m |= 1 << c
                v |= int(b) << c
            ctrl[i], cval[i] = m, v
            mats[i] = g.base_matrix()
            channel[i] = ch.get(model.gate_error(g.name, g.qubits), g.qubits)
    e = EncodedNoise()
    e.n_qubits, e.n_gates = N, G
    e.target, e.ctrl_mask, e.ctrl_value = target, ctrl, cval
    m = np.empty((G, 8))
    m[:, 0::2] = mats.reshape(G, 4).real
    m[:, 1::2] = mats.reshape(G, 4).imag
    e.matrix = m
    e.channel = channel
    e.cum = np.array(ch.cum).reshape(-1, MAX_PAULIS)
    e.n_paulis = np.array(ch.n, dtype=np.int32)
    e.chan_qubits = np.array(ch.qubits, dtype=np.int32).reshape(-1, 2)
    e.err_n_stages = np.array(ch.err_n, dtype=np.int32)
    e.err_kind = np.array(ch.err_kind, dtype=np.int32).reshape(-1, MAX_STAGES)
    e.err_index = np.array(ch.err_index, dtype=np.int32).reshape(-1, MAX_STAGES)
    e.kraus_ops = np.array(ch.kops).reshape(-1, MAX_KRAUS, 8)
    e.kraus_n_ops = np.array(ch.kn, dtype=np.int32)
    e.kraus_qubit = np.array(ch.kq, dtype=np.int32)
    e.kraus = ch.kraus
    e.n_clbits = prog.n_clbits
    e.clbit_map = np.full(prog.n_clbits, -1, dtype=np.int32)
    for c, q in prog.measures.items():
        e.clbit_map[c] = q
    e.readout = model.readout_table(prog)
    e.gate_noisy = bool((channel >= 0).any())
    e.readout_noisy = bool(e.readout.any())
    return e
