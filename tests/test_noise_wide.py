"""Noisy trajectories at 9-13 qubits against the exact density-matrix law: random entangling programs with controls
anywhere, 2-qubit Pauli errors and Kraus stages on qubits >= 8, warp-mode (<= 10 qubits) and CTA-mode (11-13)
circuits in one call, both precisions, both routes (qcm_run_noisy_small and qcm_run_noisy_small_kraus).

The law is tests/density_oracle.py's (Pauli route) or test_noise_kraus.law_rho (Kraus route) on their torch
backend, on the GPU above 10 qubits.  A 13-qubit key has too many outcomes for a useful full-key TV bound (about
0.10 at 2^18 shots), so every circuit is checked on marginals of at most 6 clbits (bound about 0.011): its 6
highest measured qubits, its 6 lowest, each measured pair a 2-qubit error on a qubit >= 8 touches, and the whole key
when it has at most 10 bits.  alpha = 1e-6 is split over all windows of a call.

A power guard keeps these checks from going vacuous: laws of mutated noise (no error after gates on qubits >= 8,
2-qubit errors mirrored, controls on qubits >= 8 dropped, readout flips read from the other row, Kraus stages on
qubits >= 8 replaced by the identity) must sit at least twice the bound from the true law on some checked window of
some circuit, at every width.  Up to 10 qubits the guard runs on the CPU, above that on the GPU."""
import functools

import numpy as np
import pytest

import density_oracle as dm
from conftest import has_cuda
from test_noise import counts_vec, random_program, reference_noise, weissman_tv_bound
from test_noise_kraus import Model, error_super, law_rho, mixed_model
from qcmrf_b200 import B200Simulator, ir
from qcmrf_b200.noise import PauliError, ReadoutError, pauli_error


def gpu(test):
    return pytest.mark.gpu(pytest.mark.skipif(not has_cuda(), reason='needs a CUDA device')(test))


HIGH = 8                                    # qubits from here up: beyond the numpy law's reach before this file
WIDE = (9, 10, 11, 12, 13)
GATE_COUNTS = (65, 33, 32, 31)              # around the kernel's 32-gate staging chunk
SHOTS = 1 << 18
ALPHA = 1e-6
PATH = {'pauli': 'noisy_trajectories', 'kraus': 'noisy_trajectories_kraus'}


# ------------------------------------------------------------------------------------------------------ circuits
def _pinned(N):
    """Gates every wide circuit carries: 2-qubit errors on a high pair, and at 13 qubits the Pauli model's
    qubit-specific errors on qubit 12 and on the pairs (12, 9) and (9, 12)."""
    g = [ir.Gate('cx', (N - 1, N - 2), (), (1,)), ir.Gate('cz', (N - 3, N - 1), (), (1,)), ir.Gate('sx', (N - 1,))]
    if N == 13:
        g += [ir.Gate('cx', (12, 9), (), (1,)), ir.Gate('ry', (12,), (0.9,)), ir.Gate('cp', (9, 12), (1.1,), (1,))]
    return g


def _wide_program(rng, N, n_gates):
    pins = _pinned(N)
    p = random_program(rng, N, n_gates - len(pins))
    for g in pins:
        p.gates.insert(int(rng.randint(len(p.gates) + 1)), g)
    return p


@functools.lru_cache(maxsize=None)
def circuits():
    """One call's circuits: 4 per width of 9-13 qubits, two small ones, and two (10 and 13 qubits) whose clbit map
    permutes the qubits, measures N - 2 of them and has more clbits than qubits."""
    rng = np.random.RandomState(9013)
    progs = [_wide_program(rng, N, n) for N in WIDE for n in GATE_COUNTS]
    progs += [random_program(rng, 3, 33), random_program(rng, 5, 40, measured=range(4))]
    for N, ncl in ((10, 14), (13, 16)):
        p = _wide_program(rng, N, 40)
        p.n_clbits = ncl
        p.measures = {int(c): int(q) for c, q in zip(rng.permutation(ncl)[:N - 2], rng.permutation(N)[:N - 2])}
        progs.append(p)
    return tuple(progs)


# -------------------------------------------------------------------------------------------------------- models
def _pauli_model():
    m = Model()
    m.nm = reference_noise(13)
    m.nm.add_quantum_error(pauli_error([('X', 0.12), ('Y', 0.06), ('I', 0.82)]), ['ry', 'sx', 'x'], [12])
    m.nm.add_quantum_error(pauli_error([('XZ', 0.09), ('IY', 0.07), ('YI', 0.03), ('II', 0.81)]), ['cx'], [12, 9])
    m.nm.add_quantum_error(pauli_error([('ZX', 0.1), ('II', 0.9)]), ['cp'], [9, 12])
    return m


@functools.lru_cache(maxsize=None)
def model(route):
    """The route's model: reference_noise with qubit-specific errors on qubit 12 and a high pair (Pauli), or
    test_noise_kraus.mixed_model, whose expanded relaxation on cx and tensored damping on cz put Kraus stages on
    both qubits of a gate (Kraus)."""
    return _pauli_model() if route == 'pauli' else mixed_model(13)


def _rho(route, prog, m, device):
    return dm.run(prog, m.nm, device) if route == 'pauli' else law_rho(prog, m, device)


@functools.lru_cache(maxsize=None)
def true_diagonal(route, i, device):
    return dm.diagonal(_rho(route, circuits()[i], model(route), device))


def true_law(route, i, device):
    return dm.key_law(circuits()[i], model(route).nm, rho=true_diagonal(route, i, device))


# ------------------------------------------------------------------------------------------------------- windows
def windows(prog, nm):
    """The clbit sets whose marginals are checked (see the module docstring)."""
    cl = {q: c for c, q in prog.measures.items()}
    by_qubit = [cl[q] for q in sorted(cl)]
    ws = {tuple(sorted(by_qubit[-6:])), tuple(sorted(by_qubit[:6]))}
    for g in prog.gates:
        if (len(g.qubits) == 2 and max(g.qubits) >= HIGH and nm.gate_error(g.name, g.qubits) is not None
                and all(q in cl for q in g.qubits)):
            ws.add(tuple(sorted(cl[q] for q in g.qubits)))
    if prog.n_clbits <= 10:
        ws.add(tuple(range(prog.n_clbits)))
    return sorted(ws)


def all_windows(route):
    ws = [windows(p, model(route).nm) for p in circuits()]
    return ws, ALPHA / sum(len(w) for w in ws)


def marginal(vec, bits):
    idx = np.arange(vec.size)
    k = np.zeros(vec.size, dtype=np.int64)
    for j, b in enumerate(bits):
        k |= ((idx >> b) & 1) << j
    return np.bincount(k, weights=vec, minlength=1 << len(bits))


def bound(law_m, alpha):
    return weissman_tv_bound(int((law_m > 0).sum()), SHOTS, alpha)


# ------------------------------------------------------------------------------------------------------- mutants
_SWAP = np.kron(np.eye(4)[[0, 2, 1, 3]], np.eye(4)[[0, 2, 1, 3]])     # 2-qubit superoperator: exchange the qubits


class _Stand:
    """An error object of a mutated model: the Kraus law reads it only through its superoperator."""


def _per_gate(m, prog, f):
    """m with each gate's error e replaced by f(gate, e, mutant) (None: no error) as a qubit-specific entry."""
    out = Model()
    out.supers = dict(m.supers)
    out.keep = []
    out.nm._all_readout, out.nm._local_readout = m.nm._all_readout, m.nm._local_readout
    for g in prog.gates:
        e = m.nm.gate_error(g.name, g.qubits)
        if e is not None and len(g.qubits) <= 2 and (g.name, tuple(g.qubits)) not in out.nm._local_gate:
            e2 = f(g, e, out)
            if e2 is not None:
                out.nm._local_gate[(g.name, tuple(g.qubits))] = e2
    return out


def _derived(out, e, key, make_pauli, make_super):
    """One mutated object per (original error, kind), kept alive with the mutant model (its id keys the law)."""
    memo = out.__dict__.setdefault('memo', {})
    if (id(e), key) not in memo:
        e2 = make_pauli() if isinstance(e, PauliError) else _Stand()
        if id(e) in out.supers:
            out.supers[id(e2)] = make_super()
        out.keep.append(e2)
        memo[(id(e), key)] = e2
    return memo[(id(e), key)]


def _no_high_errors(g, e, out):
    return None if max(g.qubits) >= HIGH else e


def _mirrored(g, e, out):
    if e.num_qubits != 2:
        return e
    return _derived(out, e, 'mirror', lambda: pauli_error([(lab[::-1], p) for lab, p in e.to_labels()]),
                    lambda: _SWAP @ out.supers[id(e)] @ _SWAP)


def _no_high_kraus(g, e, out):
    at = tuple(j for j, q in enumerate(g.qubits) if q >= HIGH)
    if not any(st[0] == 'kraus' and st[2] in at for st in e.stages):
        return e
    return _derived(out, e, at, None, lambda: error_super(e, at))


class _ControlsDropped:
    """Gate g with its controls on qubits >= HIGH ignored: the same name, qubits and error, a cache key of its own."""

    def __init__(self, g):
        keep = [j for j, q in enumerate(g.controls) if q < HIGH]
        self.name, self.qubits, self.target, self._B = g.name, g.qubits, g.target, g.base_matrix()
        self.controls = tuple(g.controls[j] for j in keep)
        self.ctrl_values = tuple(g.ctrl_values[j] for j in keep)
        self.params = tuple(g.params) + ('controls kept', tuple(keep))

    def base_matrix(self):
        return self._B

    def matrix(self):
        """On a 2-qubit gate whose one control is dropped: identity on it, the base matrix on the target."""
        assert len(self.qubits) == 2 and not self.controls
        return np.kron(self._B, np.eye(2))


def _readout_rows_swapped(nm):
    """Each qubit's assignment matrix with every row's flip probability taken from the other row (a transposed
    assignment matrix is not stochastic; this is what reading the flip of the other outcome gives)."""
    def sw(e):
        if e is None:
            return None
        a, b = e.probabilities[0, 1], e.probabilities[1, 0]
        return ReadoutError([[1 - b, b], [a, 1 - a]])
    out = Model()
    out.nm._all_gate, out.nm._local_gate = nm._all_gate, nm._local_gate
    out.nm._all_readout = sw(nm._all_readout)
    out.nm._local_readout = {q: sw(e) for q, e in nm._local_readout.items()}
    return out.nm


MUTANTS = {'pauli': ('no_error_on_high_gates', 'mirrored_2q_errors', 'high_controls_dropped', 'readout_rows_swapped'),
           'kraus': ('no_error_on_high_gates', 'mirrored_2q_errors', 'high_controls_dropped', 'readout_rows_swapped',
                     'no_kraus_on_high_qubits')}


def mutant_law(route, i, name, device):
    p, m = circuits()[i], model(route)
    if name == 'readout_rows_swapped':
        return dm.key_law(p, _readout_rows_swapped(m.nm), rho=true_diagonal(route, i, device))
    if name == 'high_controls_dropped':
        q = ir.Program(p.n_qubits, p.n_clbits, measures=dict(p.measures),
                       gates=[_ControlsDropped(g) if any(c >= HIGH for c in g.controls) else g for g in p.gates])
        return dm.key_law(p, m.nm, rho=dm.diagonal(_rho(route, q, m, device)))
    f = {'no_error_on_high_gates': _no_high_errors, 'mirrored_2q_errors': _mirrored,
         'no_kraus_on_high_qubits': _no_high_kraus}[name]
    mm = _per_gate(m, p, f)
    return dm.key_law(p, mm.nm, rho=dm.diagonal(_rho(route, p, mm, device)))


def check_power(route, widths, device):
    """Every mutant, at every width, at >= 2x the bound from the true law on some checked window."""
    progs = circuits()
    ws, alpha = all_windows(route)
    for N in widths:
        order = sorted((i for i, p in enumerate(progs) if p.n_qubits == N), key=lambda i: -len(progs[i].gates))
        todo = list(MUTANTS[route])
        for i in order:
            law = true_law(route, i, device)
            for name in list(todo):
                mut = mutant_law(route, i, name, device)
                for w in ws[i]:
                    lm = marginal(law, w)
                    if 0.5 * np.abs(marginal(mut, w) - lm).sum() >= 2 * bound(lm, alpha):
                        todo.remove(name)
                        break
            if not todo:
                break
        assert not todo, (route, N, todo)


# ------------------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize('N', [1, 3, 6, 8])
def test_torch_backend_is_the_numpy_backend(N):
    rng = np.random.RandomState(40 + N)
    nm, m = reference_noise(N), mixed_model(N)
    for _ in range(2):
        p = random_program(rng, N, 40, measured=range(N - 1) if N > 3 else None)
        a, b = dm.run(p, nm), dm.run(p, nm, device='cpu').numpy()
        assert np.abs(a - b).max() < 1e-13
        assert np.abs(dm.key_law(p, nm) - dm.key_law(p, nm, device='cpu')).max() < 1e-13
        a, b = law_rho(p, m), law_rho(p, m, device='cpu').numpy()
        assert np.abs(a - b).max() < 1e-13
        assert np.abs(dm.key_law(p, m.nm, rho=a) - dm.key_law(p, m.nm, rho=np.real(np.diag(b)))).max() < 1e-13


def test_backend_limits():
    for device, n_max in ((None, dm.MAX_QUBITS), ('cpu', dm.MAX_QUBITS_TORCH)):
        assert dm.initial_state(min(n_max, 10), device).shape == (2,) * (2 * min(n_max, 10))
        with pytest.raises(ValueError, match='at most %d qubits' % n_max):
            dm.run(ir.Program(n_max + 1, 1), device=device)


def test_circuits_cover_what_they_claim():
    progs = circuits()
    assert [p.n_qubits for p in progs[:20]] == [N for N in WIDE for _ in GATE_COUNTS]
    assert [len(p.gates) for p in progs[:20]] == list(GATE_COUNTS) * len(WIDE)
    for p in progs[:20]:
        N = p.n_qubits
        names = {g.name for g in p.gates}
        assert {'cx', 'cz', 'cp'} <= names and names & {'mcx', 'mcp'}
        assert any(max(g.controls, default=-1) >= HIGH for g in p.gates)
    assert any(p.n_clbits > p.n_qubits and len(p.measures) < p.n_qubits and
               any(c != q for c, q in p.measures.items()) for p in progs if p.n_qubits > 10)
    for route in PATH:
        ws, _ = all_windows(route)
        assert max(len(w) for wl in ws for w in wl) <= 10
        assert all(max(len(w) for w in wl) <= 6 for wl, p in zip(ws, progs) if p.n_clbits > 10)


@pytest.mark.parametrize('route', ['pauli', 'kraus'])
def test_power_guard_up_to_10_qubits(route):
    check_power(route, [9, 10], 'cpu')


# ------------------------------------------------------------------------------------------------------------ GPU
@gpu
@pytest.mark.parametrize('route', ['pauli', 'kraus'])
def test_power_guard_11_to_13_qubits(route):
    check_power(route, [11, 12, 13], 'cuda')


@gpu
@pytest.mark.parametrize('precision', ['double', 'single'])
@pytest.mark.parametrize('route', ['pauli', 'kraus'])
def test_wide_noisy_marginals_follow_the_density_matrix_law(route, precision):
    progs = circuits()
    ws, alpha = all_windows(route)
    res = B200Simulator(precision=precision, seed=1213, noise_model=model(route).nm).run(list(progs), shots=SHOTS).result()
    for i, p in enumerate(progs):
        assert res.metadata(i)['noise'] and res.metadata(i)['path'] == PATH[route], i
        obs = counts_vec(res.get_counts(i), p.n_clbits)
        assert obs.sum() == SHOTS
        law = true_law(route, i, 'cuda')
        for w in ws[i]:
            lm, om = marginal(law, w), marginal(obs, w) / SHOTS
            what = (route, precision, i, p.n_qubits, w)
            assert om[lm <= 0].sum() == 0, what
            tv = 0.5 * np.abs(om - lm).sum()
            assert tv < bound(lm, alpha), (what, tv, bound(lm, alpha))
