"""The reference-facing surface: the QCMRF mirror and the compat shims, pinned against
the programs the reference's own QCMRF.py emitted (tests/golden/ref_programs.json).
CPU only; the engine is replaced by tests/fake_native.py where a run is needed."""
import json
import os

import numpy as np
import pytest

import fake_native
from conftest import GOLDEN
from oracle import mrf as omrf, program, statevector as sv
from qcmrf_b200 import QCMRF, KL, compat, extract_probs, fidelity, ir


def test_qcmrf_validation_and_properties():
    with pytest.raises(ValueError):
        QCMRF([0, 1], [0.0] * 4)                      # not a list of lists
    with pytest.raises(ValueError):
        QCMRF([[0.0, 1.0]], [0.0] * 4)                # not ints
    with pytest.raises(ValueError):
        QCMRF([[0, 1]], [0.0] * 3)                    # wrong theta length (QCMRF.py:68-71)
    with pytest.raises(ValueError):
        QCMRF([[0, 1]], gamma=[0.1] * 5)              # wrong gamma length (QCMRF.py:73-76)
    c = QCMRF([[0, 1], [1, 2, 3]], [-0.1] * 12)
    assert (c.num_vertices, c.num_nodes, c.num_cliques, c.max_clique, c.dimension) == (4, 4, 2, 3, 12)
    assert c.num_qubits == 4 + 2 + 1 == c.num_clbits   # QCMRF.py:78
    assert c.cliques == [[0, 1], [1, 2, 3]]
    assert np.allclose(c.gamma, program.theta_to_gamma([-0.1] * 12))
    assert c.basis_gates == ['cx', 'id', 'rz', 'sx', 'x']
    ops = c.count_ops()
    assert ops['h'] == 4 + 2 * 2 and ops['x'] == 4 and ops['measure'] == 6


def test_random_default_parameters_follow_numpy_global_state():
    """No theta/gamma: theta ~ U(-5,0) from the global numpy RNG (QCMRF.py:210-213)."""
    np.random.seed(7)
    c = QCMRF([[0, 1]])
    np.random.seed(7)
    expect = [np.random.uniform(low=-5.0, high=0) for _ in range(4)]
    assert c.theta == expect


def test_host_side_postselection_helpers(aer_counts):
    Q = aer_counts['0.5'][10]
    a, b = extract_probs(Q, 2, 2), omrf.extract_probs(Q, 2, 2)
    assert np.array_equal(a[0], b[0]) and a[1] == b[1]
    P, s = extract_probs({'1000': 3}, 2, 2)
    assert s == 0 and not P.any()
    p = np.array([0.5, 0.5, 0, 0]); q = np.array([0.25, 0.25, 0.5, 0])
    assert abs(fidelity(p, q) - omrf.fidelity(p, q)) < 1e-16 and abs(KL(p, q) - omrf.kl(p, q)) < 1e-16


def test_shims_serve_only_missing_names():
    served = compat.install()
    for name in served:
        assert name in compat.SHIMMED
    import qiskit
    from qiskit import Aer, QuantumCircuit, transpile               # noqa: F401
    from qiskit.circuit.library import AND
    from qiskit.converters import circuit_to_gate                   # noqa: F401
    from qiskit.opflow import I, Z
    if getattr(qiskit, '__qcmrf_b200_shim__', False):
        assert Aer.get_backend('qasm_simulator').name() == 'qasm_simulator'
        with pytest.raises(LookupError):
            Aer.get_backend('ibmq_whatever')
        proj1 = (I - Z) / 2
        assert np.allclose(proj1.to_matrix(), np.diag([0, 1]))
        assert np.allclose(((I + Z) / 2 ^ proj1).to_matrix(), np.diag([0, 1, 0, 0]))
        a = AND(3, [1, -1, 0])
        g = ir.lower(a).gates
        assert len(g) == 1 and g[0].qubits == (0, 1, 3) and g[0].ctrl_values == (1, 0)
    import kiopto_native as px
    b = px.backend([[0, 1], [1, 2]], np.array([2, 2, 2]))
    w = px.weights(b)
    assert len(w) == 8
    th = -np.abs(np.random.RandomState(1).randn(8))
    w[:] = th
    pb, _, lnZ = omrf.brute_force_pmf([[0, 1], [1, 2]], th)
    assert abs(px.infer(b, task='partition') - lnZ) < 1e-13
    assert np.allclose([np.exp(px.logpot(b, x) - lnZ) for x in range(8)], pb)


def test_product_constructor_matches_golden_reference_programs(models):
    """The product's constructor emits the programs the reference's QCMRF.py emitted for rep 0 of every graph, and
    the oracle's restatement executes to the same state."""
    golden = json.load(open(os.path.join(GOLDEN, 'ref_programs.json')))
    assert len(golden) == 42
    for key, want in golden.items():
        scale, j, wm = key.split('/')
        C = models[scale]['GRAPHS'][int(j)]
        th = models[scale]['THETAS'][j][0]
        assert ir.to_jsonable(ir.lower(QCMRF(C, th, with_measurements=bool(int(wm))))) == want
        # ... and the oracle's restatement executes to the same state
        prog = ir.from_jsonable(want)
        N = prog.n_qubits
        a, _ = sv.run_program(ir.to_oracle_ops(prog), N)
        b, _ = sv.run_program(program.qcmrf_program(C, th, with_measurements=bool(int(wm)))[0], N)
        assert np.abs(a - b).max() < 1e-15


def test_direct_lowering_equals_walking_the_instruction_list(models):
    """QCMRF materialises its nested instruction list lazily; the engine's direct lowering must be
    the very program the generic walk finds in `.data`, and an edited circuit must fall back."""
    from qcmrf_b200 import ir
    rng = np.random.RandomState(0)
    cases = [(C, models['0.5']['THETAS'][str(j)][0]) for j, C in enumerate(models['0.5']['GRAPHS'])]
    cases.append(([[0, 1], [1, 2]], [0.0, -0.3, 0.0, -1.0, -0.2, 0.0, -0.5, -0.1]))      # skipped (gamma ~ 0) terms
    for C, th in cases:
        for kw in ({}, {'with_measurements': False}, {'beta': 0.5}):
            fast = ir.lower(QCMRF(C, th, **kw))
            slow_c = QCMRF(C, th, **kw)
            assert slow_c.__dict__['_mrf_data'] is None
            n_inst = len(slow_c.data)                                 # materialises
            assert n_inst > 0 and slow_c._lower_program() is None
            slow = ir.lower(slow_c)
            assert fast.n_qubits == slow.n_qubits and fast.n_clbits == slow.n_clbits
            assert fast.measures == slow.measures
            assert len(fast.gates) == len(slow.gates)
            for a, b in zip(fast.gates, slow.gates):
                assert (a.name, a.qubits, a.ctrl_values) == (b.name, b.qubits, b.ctrl_values)
                assert np.allclose(a.params, b.params, rtol=0, atol=0)
    # gamma-only construction and an edited circuit
    c = QCMRF([[0, 1]], gamma=[0.1, 0.2, 0.3, 0.4], with_measurements=False)
    c.h(0)
    assert ir.lower(c).gates[-1].name == 'h' and len(ir.lower(c).gates) == len(ir.lower(QCMRF([[0, 1]], gamma=[0.1, 0.2, 0.3, 0.4])).gates) + 1


def test_native_counts_formatter_equals_numpy():
    """csrc/qcm_host.c (one dict insert per distinct key, CPython C API) == the numpy formatter: same keys
    in the same (ascending) order, same counts; widths 1..64, empty input."""
    from qcmrf_b200 import build
    from qcmrf_b200.backend import _host, _keys_to_counts
    build.build_host()
    assert _host(), '_qcm_host.so did not load'
    rng = np.random.default_rng(3)
    for width, n in ((1, 50), (3, 1000), (10, 10000), (34, 10000), (63, 500), (64, 500), (34, 0)):
        hi = (1 << width) - 1
        keys = rng.integers(0, hi, size=n, dtype=np.uint64, endpoint=True) if n else np.zeros(0, dtype=np.uint64)
        if n > 10:
            keys[: n // 3] = keys[n // 3: 2 * (n // 3)]
            keys[-1] = hi
        a = _keys_to_counts(keys, width, use_native=True)
        b = _keys_to_counts(keys, width, use_native=False)
        assert type(a) is type(b) and list(a.items()) == list(b.items())
        assert sum(a.values()) == n and all(len(k) == width for k in a)


def test_sweep_grouping_through_a_batched_handle(monkeypatch):
    """A list of same-structure circuits (a beta sweep) goes through ONE batched handle: results equal the
    one-by-one path, the post-selected vectors stay "on the device" until asked for, mixed lists still work."""
    import fake_native
    from oracle import mrf
    from qcmrf_b200 import B200Simulator
    from qcmrf_b200.backend import _ResidentProbs
    fake_native.install(monkeypatch)
    monkeypatch.setattr(fake_native, 'small_max_qubits', lambda precision='double': 4)
    import qcmrf_b200._native as nat
    monkeypatch.setattr(nat, 'small_max_qubits', lambda precision='double': 4)
    C = [[0, 1], [1, 2], [2, 3]]
    rng = np.random.RandomState(5)
    th = list(-np.abs(rng.randn(12)) * 0.5)
    betas = [0.25, 0.5, 1.0, 2.0, 3.0]
    other = QCMRF([[0, 1, 2], [2, 3]], list(-np.abs(rng.randn(12))))
    for width in ('release', 'full'):
        sim = B200Simulator(precision='double', width=width, seed=3, small_batch=False)
        circs = [QCMRF(C, th, beta=b) for b in betas] + [other]
        res = sim.run(circs, shots=2000).result()
        assert [res.metadata(i)['path'] for i in range(6)] == ['sweep'] * 5 + ['statevector']
        assert isinstance(res.results()[0]['probs'], _ResidentProbs)
        for i, b in enumerate(betas):
            p, d = res.postselected_probabilities(i)
            pb, db, _ = mrf.brute_force_pmf(C, th, beta=b)
            assert np.abs(p - pb).max() < 1e-12 and abs(d - db) < 1e-12
            counts = res.get_counts(i)
            assert sum(counts.values()) == 2000 and all(len(k) == 8 and k[8 - 1 - 4] == '0' for k in counts)
        p, d = res.postselected_probabilities(5)
        pb, db, _ = mrf.brute_force_pmf([[0, 1, 2], [2, 3]], other.theta)
        assert np.abs(p - pb).max() < 1e-12
        # pmf=True copies everything, pmf=False computes delta only; chunks of 2 + 3 points
        sim.sweep_bytes = 2 * (16 << res.metadata(0)['n_phys'])
        res2 = sim.run(circs[:5], shots=0, pmf=True).result()
        assert all(isinstance(e['probs'], np.ndarray) for e in res2.results())
        assert sorted(e['meta']['sweep_points'] for e in res2.results()) == [2, 2, 3, 3, 3]
        for i, b in enumerate(betas):
            pb, db, _ = mrf.brute_force_pmf(C, th, beta=b)
            assert np.abs(res2.postselected_probabilities(i)[0] - pb).max() < 1e-12
        sim.close()


def test_px_shim_is_memoised_and_matches_the_oracle():
    """eval.py:84-93 calls px.infer once and px.logpot 2^n times per model: the stand-in evaluates one state per
    logpot call (no O(4^n) loop) and memoises ln Z per weight vector."""
    from oracle import mrf
    from qcmrf_b200.compat.shim import kiopto_native as px
    C = [[0, 1, 2], [2, 3], [4], [3, 4, 0, 1]]
    rng = np.random.RandomState(2)
    th = -np.abs(rng.randn(8 + 4 + 2 + 16))
    b = px.backend(C, np.array([2] * 5))
    assert len(px.weights(b)) == 30
    px.weights(b)[:] = th
    lz = px.infer(b, task='partition')
    calls = []
    orig = b.energies
    b.energies = lambda: calls.append(1) or orig()
    p = np.array([np.exp(px.logpot(b, x) - px.infer(b, task='partition')) for x in range(32)])
    assert not calls                                            # neither logpot nor the memoised infer enumerates again
    pb, _db, _ = mrf.brute_force_pmf(C, th)
    assert np.abs(p - pb).max() < 1e-14
    px.weights(b)[0] -= 1.0                                     # new weights: ln Z is recomputed
    assert px.infer(b, task='partition') != lz


def test_vectorised_sweep_preparation_equals_one_by_one(monkeypatch):
    """The vectorised release-width preparation of a same-graph QCMRF list yields the tables the per-circuit
    lower/fuse/plan path yields (projection factors, released-qubit probabilities), for theta/beta and gamma input."""
    import fake_native
    from qcmrf_b200 import B200Simulator, workloads
    fake_native.install(monkeypatch)
    sim = B200Simulator(precision='double', width='release', small_batch=False)
    C = workloads.chain(14)
    th = workloads.theta_for(C, seed=2)
    circs = [QCMRF(C, th, beta=(j + 1) / 8.0) for j in range(9)]
    fast = sim._qcmrf_release_sweep(circs, None, 'double')
    assert fast is not None
    slow = sim._stack_sweep([sim.prepare(QCMRF(C, th, beta=(j + 1) / 8.0)) for j in range(9)])
    assert np.array_equal(fast.ops, slow.ops) and np.array_equal(fast.proj_ops, slow.proj_ops)
    assert np.allclose(fast.tables, slow.tables, rtol=0, atol=0)
    assert np.allclose(fast.proj_tables, slow.proj_tables, rtol=1e-14, atol=0)
    assert np.allclose(fast.p1, slow.p1, rtol=1e-14, atol=1e-300)
    for a, b in zip(fast.released, slow.released):
        assert np.array_equal(np.asarray(a), np.asarray(b))
    # gamma input, and a list the shortcut must refuse (a skipped term changes the program structure)
    g = [0.1 + 0.01 * k for k in range(4 * 13)]
    fast = sim._qcmrf_release_sweep([QCMRF(C, gamma=g), QCMRF(C, gamma=[x * 0.5 for x in g])], None, 'double')
    slow = sim._stack_sweep([sim.prepare(QCMRF(C, gamma=g)), sim.prepare(QCMRF(C, gamma=[x * 0.5 for x in g]))])
    assert np.allclose(fast.proj_tables, slow.proj_tables, rtol=1e-14, atol=0) and np.allclose(fast.p1, slow.p1, rtol=1e-14)
    th0 = list(th); th0[5] = 0.0
    assert sim._qcmrf_release_sweep([QCMRF(C, th), QCMRF(C, th0)], None, 'double') is None


def test_list_of_large_circuits_is_a_pipeline_with_identical_results(monkeypatch, models):
    """run(list) on the large-state path enqueues circuit i+1 before collecting circuit i (execute_deferred: a ring of
    three result buffers, qcm_mark / qcm_wait tickets).  Host logic on the emulator: results equal one blocking run() per
    circuit with the same Philox stream, across a change of state size inside the list; the ring refuses a fourth
    pending execution and a second collection."""
    import fake_native
    fake_native.install(monkeypatch)
    from qcmrf_b200 import QCMRF, B200Simulator
    items = []
    for j, t in ((1, 0), (1, 1), (3, 0), (1, 2), (5, 0), (5, 1), (5, 2), (5, 3), (1, 3)):
        items.append((models['0.5']['GRAPHS'][j], models['0.5']['THETAS'][str(j)][t]))
    sim = B200Simulator(precision='double', small_batch=False, sweep_batch=False, seed=3)
    calls = []
    orig = sim.execute_deferred
    monkeypatch.setattr(sim, 'execute_deferred', lambda *a, **k: (calls.append(a[0]), orig(*a, **k))[1])
    res = sim.run([QCMRF(c, th) for c, th in items], shots=3000).result()
    assert len(calls) == len(items)                                    # every circuit went through the pipeline
    one = B200Simulator(precision='double', small_batch=False, sweep_batch=False, seed=3)
    for i, (c, th) in enumerate(items):
        r1 = one.run(QCMRF(c, th), shots=3000, stream_ids=[i]).result()
        assert r1.get_counts() == res.get_counts(i), i
        p1, d1 = r1.postselected_probabilities(0)
        p, d = res.postselected_probabilities(i)
        assert np.array_equal(p, p1) and d == d1, i
        assert abs(p.sum() - 1.0) < 1e-12 and res.postselected_probabilities(i)[0] is p      # normalised once, in the pipeline
        assert res.metadata(i)['philox_stream'] == i and res.metadata(i)['path'] == 'statevector'
    pr = sim.prepare(QCMRF(*items[0]))
    fins = [sim.execute_deferred(pr, 50, seed=1, stream=s) for s in range(3)]
    with pytest.raises(RuntimeError):
        sim.execute_deferred(pr, 50, seed=1, stream=3)
    outs = [f() for f in fins]
    with pytest.raises(RuntimeError):
        fins[1]()
    k0, p0, m0 = sim.execute(pr, 50, seed=1, stream=0)
    assert np.array_equal(outs[0][0], k0) and np.array_equal(outs[0][1], p0) and outs[0][2] == m0
    # results handed out are copies: the ring slot is reused by the fourth execution without changing them
    keep = outs[0][0].copy()
    sim.execute_deferred(pr, 50, seed=1, stream=9)()
    assert np.array_equal(outs[0][0], keep)
    # another state size while an execution is pending would release the state under it: refused until collected
    other = sim.prepare(QCMRF(*items[2]))
    assert other.plan.n_phys != pr.plan.n_phys
    fin = sim.execute_deferred(pr, 50, seed=1, stream=0)
    with pytest.raises(RuntimeError, match='pending'):
        sim.execute_deferred(other, 50, seed=1, stream=0)
    assert np.array_equal(fin()[0], k0)
    sim.execute_deferred(other, 50, seed=1, stream=0)()
    # no shots / release width: the blocking path answers through the same callable
    k, p, m = sim.execute_deferred(pr, 0)()
    assert k is None and np.array_equal(p, p0) and m == m0


@pytest.mark.parametrize('seed', range(3))
def test_random_generic_circuits_through_the_public_call(monkeypatch, seed):
    """Seeded fuzz of the generic front end through B200Simulator.run on the emulator: random circuits over the whole gate
    surface (plain and transpiled to cx/id/rz/sx/x), a random subset of qubits measured into shuffled clbits, a random
    variable-register width -- post-selected pmf and success probability against an independent textbook simulation,
    keys only where the exact key distribution has mass, histogram within its Weissman bound; every fusion mode, the
    batched-small and the large-state path, full and release width."""
    import fake_native
    fake_native.install(monkeypatch)
    from test_host_fusion import _random_circuit, _textbook_state
    from qcmrf_b200 import B200Simulator, transpile
    from qcmrf_b200.circuit import QuantumCircuit
    rng = np.random.RandomState(9100 + seed)
    checked = 0
    for trial in range(8):
        nq = int(rng.randint(1, 6))
        base = _random_circuit(rng, nq, int(rng.randint(1, 24)))
        pw = np.abs(_textbook_state(base)) ** 2
        nv = int(rng.randint(1, nq + 1))
        mq = [int(q) for q in rng.permutation(nq)[:int(rng.randint(1, nq + 1))]]
        cbits = [int(b) for b in rng.permutation(len(mq))]
        c = QuantumCircuit(nq, len(mq))
        for ins in base.data:
            c._qc_add(ins.operation, list(ins.qubits))
        for q, b in zip(mq, cbits):
            c.measure(q, b)
        if trial % 2:
            c = transpile(c, basis_gates=['cx', 'id', 'rz', 'sx', 'x'])
        kept = pw[:1 << nv].sum()
        if kept < 1e-9:
            continue
        idx = np.arange(1 << nq)
        key = np.zeros_like(idx)
        for q, b in zip(mq, cbits):
            key |= ((idx >> q) & 1) << b
        kp = np.bincount(key, weights=pw, minlength=1 << len(mq))
        bound = 0.5 * np.sqrt(2 * ((1 << len(mq)) * np.log(2) + np.log(1e7)) / 2000)
        for fus, small, width in (('off', True, 'full'), ('clique', False, 'full'), ('blocked', False, 'release'),
                                  ('blocked', True, 'full')):
            sim = B200Simulator(precision='double', fusion=fus, small_batch=small, width=width, seed=1)
            res = sim.run(c, shots=2000, n_vars=nv).result()
            p, d = res.postselected_probabilities(0)
            assert np.abs(p - pw[:1 << nv] / kept).max() < 1e-10 and abs(d - kept) < 1e-10, (seed, trial, fus, small, width)
            cnt = res.get_counts()
            assert sum(cnt.values()) == 2000 and all(len(k) == len(mq) and kp[int(k, 2)] > 1e-14 for k in cnt)
            emp = np.zeros(1 << len(mq))
            for k, v in cnt.items():
                emp[int(k, 2)] = v / 2000
            assert 0.5 * np.abs(emp - kp).sum() < bound, (seed, trial, fus, small, width)
            checked += 1
    assert checked >= 16


def test_pipelined_list_with_equal_state_size_and_other_pmf_size(monkeypatch):
    """Two circuits with the same number of stored qubits but different variable counts: the pipeline of run() must
    collect the first before the second needs result buffers of another size.  Counts, pmf and success probability
    equal one run() per circuit with the same Philox stream."""
    import fake_native
    fake_native.install(monkeypatch)
    from qcmrf_b200 import B200Simulator
    rng = np.random.RandomState(12)
    a = QCMRF([[0, 1], [1, 2], [2, 3], [3, 4]], list(-np.abs(rng.randn(16)) * 0.5))
    b = QCMRF([[0, 1], [1, 2], [2, 3], [0, 3], [0, 2]], list(-np.abs(rng.randn(20)) * 0.5))
    sim = B200Simulator(precision='double', small_batch=False, sweep_batch=False, seed=4)
    assert sim.prepare(a).plan.n_phys == sim.prepare(b).plan.n_phys
    circs = [a, b, a, b]
    res = sim.run(circs, shots=1500).result()
    one = B200Simulator(precision='double', small_batch=False, sweep_batch=False, seed=4)
    for i, c in enumerate(circs):
        r1 = one.run(c, shots=1500, stream_ids=[i]).result()
        assert res.get_counts(i) == r1.get_counts(), i
        p, d = res.postselected_probabilities(i)
        p1, d1 = r1.postselected_probabilities(0)
        assert np.array_equal(p, p1) and d == d1, i


def test_sweep_chunks_respect_the_engine_batch_limit(monkeypatch):
    """A sweep whose points would fit sweep_bytes many times over is still cut into chunks of at most 65 535 points,
    the most one batched handle takes."""
    import fake_native
    fake_native.install(monkeypatch)
    from qcmrf_b200 import B200Simulator
    SWEEP_MAX_POINTS = 65535                            # qcm_create_batched refuses more points
    sim = B200Simulator(precision='single', small_batch=False, seed=1)
    c = QCMRF([[0, 1], [1, 2]], [-0.3] * 8)
    pr = sim.prepare(c)
    n = 70000
    sim.sweep_bytes = 1 << 40                           # state room for ~2^28 points: only the batch limit applies
    chunks = []

    class _T:
        def timing(self):
            return dict(sample_ms=0.0, postselect_ms=0.0)

    def fake_execute_sweep(sw, shots, seed, streams, precision, pmf, first, B):
        assert 2 <= B <= SWEEP_MAX_POINTS and len(streams) == B
        chunks.append((first, B))
        sim._last = _T()
        return None, None, np.full(B, 0.5)
    monkeypatch.setattr(sim, 'execute_sweep', fake_execute_sweep)
    out = sim._run_sweep([c] * n, [pr] * n, 0, 1, np.arange(n), 'single', False)
    assert len(out) == n and sum(B for _f, B in chunks) == n
    assert chunks[0] == (0, SWEEP_MAX_POINTS) and chunks[1] == (SWEEP_MAX_POINTS, n - SWEEP_MAX_POINTS)


def test_variables_that_are_never_stored(monkeypatch):
    """A circuit whose highest variable qubits are never touched stores fewer qubits than it has variables: the
    large-state path post-selects over the stored ones and pads the pmf with the never-stored qubits' |0>."""
    import fake_native
    fake_native.install(monkeypatch)
    from qcmrf_b200 import B200Simulator
    from qcmrf_b200.circuit import QuantumCircuit
    c = QuantumCircuit(4, 4)
    c.h(0)
    c.ry(0.7, 1)
    c.cx(0, 1)
    c.measure(range(4), range(4))
    sim = B200Simulator(precision='double', small_batch=False, seed=2)
    assert sim.prepare(c, n_vars=4).plan.n_phys < 4
    a = np.array([np.cos(0.35), np.sin(0.35)])
    want = np.zeros(16)
    for x0 in (0, 1):
        for x1 in (0, 1):
            want[x0 | ((x1 ^ x0) << 1)] = 0.5 * a[x1] ** 2
    for circs in (c, [c, c]):
        res = sim.run(circs, shots=500, n_vars=4).result()
        p, d = res.postselected_probabilities(0)
        assert np.abs(p - want).max() < 1e-12 and abs(d - 1.0) < 1e-12
