"""Pauli gate errors and readout errors for noisy shot simulation (Aer's names and conventions).

    from qcmrf_b200.noise import NoiseModel, depolarizing_error, ReadoutError
    nm = NoiseModel()
    nm.add_all_qubit_quantum_error(depolarizing_error(1e-3, 1), ['sx', 'x', 'id'])
    nm.add_all_qubit_quantum_error(depolarizing_error(1e-2, 2), ['cx'])
    nm.add_all_qubit_readout_error(ReadoutError([[0.98, 0.02], [0.02, 0.98]]))
    counts = B200Simulator(noise_model=nm).run(circuits, shots=10000).result().get_counts()

Semantics (as Aer): every gate is applied and then its error channel acts on the gate's qubits; measurements are
deferred to the end of the program; each measured clbit is flipped by its measured qubit's readout error.  Every
shot is an independent trajectory with its own Pauli draws, outcome and readout draws, so the counts are i.i.d.
samples of the density-matrix law.

Errors attach to the primitive gates the circuit lowers to (qcmrf_b200.ir): a ``swap`` is three ``cx`` and a
composite instruction is its definition's gates, so errors are given for primitive gate names only.
"""
import numpy as np

from . import ir

__all__ = ['PauliError', 'pauli_error', 'depolarizing_error', 'ReadoutError', 'NoiseModel']

_PAULI_CODE = {'I': 0, 'X': 1, 'Y': 2, 'Z': 3}
#: gate names lowering keeps as primitives, with their qubit count (None: any, the multi-controlled gates)
_ARITY = dict([(n, 1) for n in list(ir._ONEQ) + list(ir._PARAM1Q) + ['u']] +
              [(n, 2) for n in ir._CTRL_BASE if n not in ('mcx', 'mcp')] + [('mcx', None), ('mcp', None)])
#: most Pauli terms of one channel (a 2-qubit error)
MAX_PAULIS = 16


class PauliError:
    """A Pauli channel on 1 or 2 qubits: rho -> sum_k p_k P_k rho P_k.

    ``probs[k]`` is the probability of the Pauli whose code on the channel's qubit j is ``(k >> 2j) & 3``
    (0 = I, 1 = X, 2 = Y, 3 = Z); k = 0 is the identity."""

    def __init__(self, n_qubits, probs):
        self.num_qubits = int(n_qubits)
        self.probs = np.asarray(probs, dtype=np.float64)
        self.probs.setflags(write=False)

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
    if not isinstance(error, PauliError):
        raise ValueError('only Pauli errors (pauli_error, depolarizing_error) are supported, got %r' % (error,))


class NoiseModel:
    """Gate errors keyed by (gate name, qubits) and readout errors keyed by qubit.  A qubit-specific entry wins over
    the all-qubit one; a second error for the same key is refused (errors are not composed)."""

    def __init__(self):
        self._all_gate = {}          # name -> PauliError
        self._local_gate = {}        # (name, qubits tuple) -> PauliError
        self._all_readout = None
        self._local_readout = {}     # qubit -> ReadoutError

    def __repr__(self):
        return 'NoiseModel(gates=%s, readout=%s)' % (sorted(set(self._all_gate) | {k[0] for k in self._local_gate}),
                                                     'all' if self._all_readout is not None else sorted(self._local_readout))

    def is_ideal(self):
        """True when no error of the model has a non-identity probability above 0."""
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
        """The PauliError that follows gate `name` on `qubits` (controls..., target), or None."""
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
    2x2 matrix (fp64, row-major re/im) and a channel index (-1: no error); one record per
    channel: cumulative Pauli probabilities and the gate's qubits."""
    __slots__ = ('n_qubits', 'n_gates', 'target', 'ctrl_mask', 'ctrl_value', 'matrix', 'channel', 'cum', 'n_paulis',
                 'chan_qubits', 'clbit_map', 'readout', 'gate_noisy', 'readout_noisy', 'n_clbits')

    @property
    def noisy(self):
        return self.gate_noisy or self.readout_noisy


class _Channels:
    def __init__(self):
        self.index = {}
        self.cum, self.n, self.qubits = [], [], []

    def get(self, err, qubits):
        """Channel index of `err` on `qubits` (-1 for an error that never applies)."""
        if err is None or err.ideal():
            return -1
        if len(qubits) > 2:
            raise ValueError('an error is attached to a gate on %d qubits: transpile first' % len(qubits))
        if len(qubits) != err.num_qubits:
            raise ValueError('a %d-qubit error cannot follow a gate on qubits %r' % (err.num_qubits, tuple(qubits)))
        key = (id(err), tuple(qubits))
        k = self.index.get(key)
        if k is None:
            k = self.index[key] = len(self.cum)
            c = np.zeros(MAX_PAULIS)
            c[:err.probs.size] = np.cumsum(err.probs)
            c[err.probs.size - 1:] = 1.0              # the last entry catches every uniform in [0, 1)
            self.cum.append(c)
            self.n.append(err.probs.size)
            self.qubits.append((qubits[0], qubits[1] if len(qubits) > 1 else -1))
        return k


def encode(prog, model):
    """Encode a lowered Program (an ir.BasisProgram straight from its arrays) with the errors `model` attaches to
    its gates.  Raises ValueError for an error on a gate of 3 or more qubits ("transpile first")."""
    N = prog.n_qubits
    ch = _Channels()
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
    e.n_clbits = prog.n_clbits
    e.clbit_map = np.full(prog.n_clbits, -1, dtype=np.int32)
    for c, q in prog.measures.items():
        e.clbit_map[c] = q
    e.readout = model.readout_table(prog)
    e.gate_noisy = bool((channel >= 0).any())
    e.readout_noisy = bool(e.readout.any())
    return e
