"""Qiskit-style backend over the CUDA engine.

Drop-in for the call the reference makes (/root/reference/run_experiment.py:54-57):

    simulator = Aer.get_backend('qasm_simulator')
    result = simulator.run(T, shots=SHOTS).result()
    counts = result.get_counts()

``run`` accepts one circuit or a list, transpiled (cx/id/rz/sx/x) or not, with or
without measurements, and returns counts keyed exactly as Aer does (clbit N-1
leftmost, one register, unmeasured clbits '0').  Beyond Aer's surface it offers the
exact post-selected probability vector the reference otherwise estimates from
counts (QCMRF.py:263-284, eval.py:115-123): ``Result.postselected_probabilities``
and ``B200Simulator.exact``.

All amplitude arithmetic, the post-selection reduction and the shot sampling run on
the GPU through the C ABI (include/qcmrf_b200.h); this file only lowers, fuses,
plans and formats.
"""
import copy
import os
import time
from typing import List, Optional, Sequence

import numpy as np

from . import _native, fusion, ir, plancache

__all__ = ['B200Simulator', 'Job', 'Result', 'Counts']

_FUSION_MODES = ('off', 'clique', 'blocked')
#: most sweep points one batched handle holds (the engine's limit: they are the grid's y dimension)
SWEEP_MAX_POINTS = 65535


class Counts(dict):
    """get_counts() value: {bitstring: int}; plain-dict compatible (json.dumps works)."""

    def shots(self):
        return sum(self.values())

    def int_outcomes(self):
        return {int(k, 2): v for k, v in self.items()}

    def most_frequent(self):
        return max(self.items(), key=lambda kv: kv[1])[0]


class _Prepared:
    __slots__ = ('prog', 'fc', 'plan', 'clbit_map', 'n_vars', 'ps', 'name', 'virtual', 'proj', '_released_tabs')


class _Sweep:
    """Circuits with ONE program structure (a theta / beta sweep over one graph), stacked for a batched handle:
    shared ops, per-point coefficient tables as rows."""
    __slots__ = ('prs', 'ops', 'tables', 'proj_ops', 'proj_tables', 'released', 'p1', 'n_phys', 'ps', 'clbit_map', 'n_vars')


class _ResidentProbs:
    """A post-selected block that was left on the GPU (sweeps: 2^n doubles per point add up quickly); fetched on
    first use, valid until the handle's next post-selection."""
    __slots__ = ('handle', 'generation', 'point', 'n_bits', 'value')

    def __init__(self, handle, point, n_bits):
        self.handle, self.generation, self.point, self.n_bits, self.value = handle, handle.generation, point, n_bits, None

    def get(self):
        if self.value is None:
            if self.handle.generation != self.generation or not self.handle._h:
                raise RuntimeError('the post-selected vector of this sweep point is no longer resident on the GPU (a later run '
                                   'reused the state); run the sweep with pmf=True to copy every vector to the host')
            self.value = self.handle.fetch_probs(self.point, self.n_bits)
        return self.value


_host_lib = None


def _host():
    """qcmrf_b200/_qcm_host.so (csrc/qcm_host.c, CPython C API), or False when it is not built."""
    global _host_lib
    if _host_lib is None:
        import ctypes
        path = os.path.join(os.path.dirname(os.path.abspath(__file__)), '_qcm_host.so')
        try:
            L = ctypes.PyDLL(path)
            L.qcm_counts_dict.restype = ctypes.py_object
            L.qcm_counts_dict.argtypes = [ctypes.c_void_p, ctypes.c_ssize_t, ctypes.c_int]
            vp = ctypes.c_void_p
            L.qcm_released_keys.restype = ctypes.c_int
            L.qcm_released_keys.argtypes = [vp, ctypes.c_int64, vp, ctypes.c_int, vp, vp, ctypes.c_int, vp, vp, vp, vp,
                                            ctypes.c_int, vp]
            _host_lib = L
        except OSError:
            _host_lib = False
    return _host_lib


def _clone_plan(pl, tables, fc):
    """A cached plan around fresh coefficient tables (plancache.PlanCache rebuild hook)."""
    q = copy.copy(pl)
    q.tables = tables[0]
    q.global_phase = fc.global_phase
    return q


def _keys_to_counts(keys, width, use_native=True):
    """uint64 keys -> Counts with Aer's key format (clbit width-1 leftmost), keys in ascending order.
    Native formatter (sort, run lengths, one dict insert per distinct key) when built; the numpy
    version below gives the same dict (tests/test_circuit_api.py)."""
    width = max(int(width), 1)
    L = _host() if (use_native and width <= 64) else False
    if L:
        k = np.ascontiguousarray(keys, dtype=np.uint64)
        return Counts(L.qcm_counts_dict(k.ctypes.data, k.size, width))
    vals, cnt = np.unique(np.asarray(keys, dtype=np.uint64), return_counts=True)
    bits = np.unpackbits(vals.astype('>u8').view(np.uint8).reshape(-1, 8), axis=1)[:, 64 - width:] if width <= 64 else None
    if bits is None:
        fmt = '0%db' % width
        return Counts({format(int(v), fmt): int(c) for v, c in zip(vals, cnt)})
    text = (bits + np.uint8(48)).tobytes().decode('ascii')
    return Counts({text[i * width:(i + 1) * width]: c for i, c in enumerate(cnt.tolist())})


def _normalised(probs, kept):
    """The post-selected pmf from the engine's unnormalised block, IN PLACE (the block is the caller's own copy): inside a
    pipelined list this runs while the GPU works on the next circuit; a fresh 1 MiB quotient per circuit at the end of the
    call costs 0.4 ms each in page faults alone.  None when there is nothing to normalise."""
    if probs is None or kept is None or not isinstance(probs, np.ndarray) or not probs.flags.writeable:
        return None
    if kept > 0:
        np.divide(probs, kept, out=probs)
    return probs


class Result:
    def __init__(self, entries, single, backend_name, seed, shots, time_taken):
        self._entries = entries
        self._single = single
        self.backend_name = backend_name
        self.seed = seed
        self.shots = shots
        self.time_taken = time_taken
        self.success = True

    def _idx(self, i):
        if i is None:
            if len(self._entries) != 1:
                raise ValueError('result holds %d experiments: give an index' % len(self._entries))
            return 0
        if isinstance(i, (int, np.integer)):
            return int(i)
        for j, e in enumerate(self._entries):          # by circuit object or name
            if e['circuit'] is i or e['name'] == i:
                return j
        raise KeyError(i)

    def get_counts(self, experiment=None):
        if experiment is None:
            if self._single:
                return self._entries[0]['counts']
            return [e['counts'] for e in self._entries]
        return self._entries[self._idx(experiment)]['counts']

    def postselected_probabilities(self, experiment=None):
        """(p, delta): exact pmf over the n variable qubits conditioned on every other
        measured-out qubit being 0 (index: x_0 = MSB, as eval.py:100-101) and the success
        probability delta."""
        e = self._entries[self._idx(experiment)]
        if e.get('pmf') is not None:                        # normalised while the list's next circuit was running
            return e['pmf'], e['kept']
        if e['probs'] is None:
            raise ValueError('circuit has no known variable-register width: pass n= to exact() or run a QCMRF')
        if isinstance(e['probs'], _ResidentProbs):
            e['probs'] = e['probs'].get()                   # sweep: the vector stayed on the GPU until asked for
        kept = e['kept']
        p = e['probs'] / kept if kept > 0 else e['probs']
        return p, kept

    def success_probability(self, experiment=None):
        return self._entries[self._idx(experiment)]['kept']

    def metadata(self, experiment=None):
        return self._entries[self._idx(experiment)]['meta']

    def results(self):
        return self._entries

    def to_dict(self):
        return {'backend_name': self.backend_name, 'success': True, 'shots': self.shots, 'seed': self.seed,
                'time_taken': self.time_taken,
                'results': [{'name': e['name'], 'counts': dict(e['counts']) if e['counts'] is not None else None,
                             'success_probability': e['kept'], 'metadata': e['meta']} for e in self._entries]}


class Job:
    """Synchronous job object (the reference calls .result() immediately)."""

    def __init__(self, result):
        self._result = result

    def result(self, timeout=None):
        return self._result

    def status(self):
        return 'DONE'

    def done(self):
        return True

    def job_id(self):
        return 'qcmrf-b200-%x' % id(self)


class B200Simulator:
    """Statevector backend on one B200.

    options: precision 'double'|'single'; fusion 'off'|'clique'|'blocked';
    block_max 1..5 (targets per blocked pass), expand_max <= 8 (targets of a pass that only
    materialises new qubits); device; seed (None = fresh entropy, as
    the unseeded Aer run of the reference)."""

    def __init__(self, name='qasm_simulator', device=0, precision='double', fusion='blocked', block_max=4,
                 seed=None, small_batch=True, small_fusion='clique', width='full', expand_max=8, plan_cache=True,
                 sweep_batch=True, sweep_state_bytes=1 << 28, sweep_bytes=32 << 30):
        if fusion not in _FUSION_MODES:
            raise ValueError('fusion must be one of %r' % (_FUSION_MODES,))
        if width not in ('full', 'release'):
            raise ValueError("width must be 'full' or 'release'")
        # 'release': measure-and-release -- qubits materialised by one sweep and never used again (the
        # clique ancillas) are not stored; their outcomes are drawn from the sweep's coefficients and
        # the post-selected vector is obtained by projecting them on 0 (SURVEY.md App. E.2)
        self.width = width
        self._name = name
        self.device = device
        self.precision = precision
        self.fusion = fusion
        self.block_max = block_max
        self.expand_max = expand_max          # width of passes that only materialise new qubits (<= 8)
        self.seed = seed
        self.small_batch = small_batch
        self.small_fusion = small_fusion      # batched small circuits: fused programs are ~30x shorter to plan and ship
        self._handles = {}
        self._pinned = {}                      # page-locked result buffers of the last sweep shape
        self._ring = None                      # page-locked result buffers of execute_deferred (three slots)
        self._launches_closed = 0
        self._last = None
        self._plan_cache = plancache.PlanCache() if plan_cache else None
        self.breakdown_ms = None               # host-side split of the last large-state run (bench.py)
        # circuits of one structure in a run() list (a theta / beta sweep) whose states are at most
        # sweep_state_bytes each go through ONE batched handle (every kernel launched once for all points),
        # in chunks of at most sweep_bytes of state
        self.sweep_batch = sweep_batch
        self.sweep_state_bytes = int(sweep_state_bytes)
        self.sweep_bytes = int(sweep_bytes)

    def name(self):
        return self._name

    def __repr__(self):
        return "B200Simulator('%s', precision=%s, fusion=%s)" % (self._name, self.precision, self.fusion)

    def set_options(self, **kw):
        for k, v in kw.items():
            if not hasattr(self, k):
                raise AttributeError('unknown option %s' % k)
            setattr(self, k, v)

    # -- host-side preparation -------------------------------------------------------
    def prepare(self, circuit, n_vars=None, fusion_mode=None, block_max=None, small=False, elide=None,
                width=None) -> _Prepared:
        mode = fusion_mode or (self.small_fusion if small else self.fusion)
        width = width or self.width
        prog = ir.lower(circuit)
        if prog.n_clbits > 64:
            raise ValueError('at most 64 classical bits are supported')
        if n_vars is None:
            n_vars = prog.metadata.get('num_vertices')
        release = width == 'release' and not small
        fc = fusion.fuse(prog, 'clique' if release or mode != 'off' else 'off')
        virtual = []
        if release:
            fc, virtual = fusion.split_releasable(fc, keep_below=n_vars or 0)
        lazy = (mode == 'blocked') and not small
        bm = block_max or self.block_max
        emax = max(bm, self.expand_max) if block_max is None else block_max

        def build(f):
            p = fusion.plan(f, lazy=lazy, block_max=bm, elide=elide, expand_max=emax)
            return p, [p.tables]

        if release or self._plan_cache is None:
            pl = build(fc)[0]
        else:
            # same structure as an earlier circuit (a theta / beta sweep): reuse its plan, refresh the tables
            pl = self._plan_cache.get(fc, ('b200', lazy, bm, elide, emax), build, _clone_plan)
        pr = _Prepared()
        pr.prog, pr.fc, pr.plan = prog, fc, pl
        pr.name = prog.name
        pr.virtual, pr.proj = [], None
        if virtual:
            self._prepare_release(pr, virtual)
        pr.clbit_map = np.full(prog.n_clbits, -1, dtype=np.int32)
        for c, q in prog.measures.items():
            p = pl.layout[q]
            pr.clbit_map[c] = p if p < pl.n_phys else -1
        pr.n_vars = n_vars
        pr.ps = None
        if n_vars is not None:
            if not 0 <= n_vars <= prog.n_qubits:
                raise ValueError('n_vars out of range')
            mask = 0
            for q in range(n_vars, prog.n_qubits):
                if pl.layout[q] < pl.n_phys:
                    mask |= 1 << pl.layout[q]
            pr.ps = (mask, 0, n_vars)
        return pr

    def _prepare_release(self, pr, virtual):
        """Released sweeps: per sweep the physical index qubits and P(outcome 1 | index); and the
        diagonal passes that project every released qubit on 0 (merged, <= QCM_MAX_CTRL index bits each)."""
        pl = pr.plan
        diag = []
        for op in virtual:
            ctrl = [pl.layout[q] for q in op.ctrls]
            if any(c >= pl.n_phys for c in ctrl):
                raise ValueError('released sweep is controlled by a qubit that is never stored')
            a0, a1 = op.table[:, 0, 0], op.table[:, 1, 0]
            w0, w1 = np.abs(a0) ** 2, np.abs(a1) ** 2
            pr.virtual.append({'qubit': op.target, 'ctrl': ctrl, 'p1': w1 / (w0 + w1)})
            diag.append((ctrl, a0))
        em = fusion._Emitter()
        act = pl.final_active
        merged = [fusion.sort_diag_ctrl(c, t) for c, t in fusion.merge_diagonals(diag)]
        if len(merged) > 1:                                   # one sweep for all of them: a BLOCK without targets
            em.op(fusion.QCM_OP_BLOCK, target=0, ctrl=(), n_in=act, n_out=act, n_ctrl=len(merged))
        for ctrl, tab in merged:
            em.op(fusion.QCM_OP_DIAG, ctrl=ctrl, n_in=act, n_out=act,
                  table_off=em.table(fusion._diag_table_f64(tab)))
        pr.proj = em.finish()

    def _handle(self, n_phys, precision, batch=1):
        key = (n_phys, precision) if batch == 1 else (n_phys, precision, batch)
        h = self._handles.get(key)
        if h is None:
            if self._ring is not None and any(rec is not None and not rec['done'] for rec in self._ring['busy']):
                # the state of a pending execute_deferred() would be released under its running kernels
                raise RuntimeError('deferred executions are pending on the state that a new state size would replace: '
                                   'collect them first (call what execute_deferred returned)')
            for k in list(self._handles):              # one big state at a time
                self._launches_closed += self._handles[k].timing()['kernel_launches']
                self._handles.pop(k).close()
            h = _native.Handle(n_phys, precision, self.device, batch=batch) if batch > 1 else \
                _native.Handle(n_phys, precision, self.device)
            self._handles[key] = h
        return h

    def close(self):
        for k in list(self._handles):
            self._handles.pop(k).close()
        self._ring = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _probs_from_handle(self, h, pr):
        pl = pr.plan
        n = pr.n_vars
        # variables that are never stored (|0> throughout) lie outside the state: the general marginal below pads them
        ident = n <= pl.n_phys and all(pl.layout[q] == q for q in range(n))
        mask, value, _ = pr.ps
        if ident:
            return h.postselect(mask, value, n)
        # variables are not physical qubits 0..n-1: take the marginal on the host side
        nb = pl.n_phys
        if nb > 26:
            raise ValueError('post-selected vector needs the variable qubits on the low physical qubits')
        full, kept = h.postselect(mask, value, nb)
        idx = np.arange(1 << nb)
        out_idx = np.zeros(1 << nb, dtype=np.int64)
        for q in range(n):
            out_idx |= ((idx >> pl.layout[q]) & 1) << q
        probs = np.zeros(1 << n)
        np.add.at(probs, out_idx, full)
        return probs, kept

    # -- public API ---------------------------------------------------------------------
    def run(self, circuits, shots=1024, seed=None, precision=None, n_vars=None, stream_ids=None, pmf=None, **options):
        """stream_ids: Philox stream per circuit (default: its index in the list) -- a batch split over
        several GPUs passes the global indices so that the counts do not depend on the partition.
        pmf: sweeps only (circuits of one structure run through one batched handle) -- True copies every point's
        post-selected vector to the host, None (default) leaves them on the GPU until
        Result.postselected_probabilities(i) asks for one, False computes only delta."""
        t0 = time.perf_counter()
        single = not isinstance(circuits, (list, tuple))
        circs = [circuits] if single else list(circuits)
        precision = precision or self.precision
        if seed is None:
            seed = self.seed
        if seed is None:
            seed = int.from_bytes(os.urandom(8), 'little')
        shots = int(shots)
        small_max = _native.small_max_qubits(precision)
        entries = [None] * len(circs)
        sid = (lambda i: i) if stream_ids is None else (lambda i: int(stream_ids[i]))
        small_ids, small_prep = [], []
        large = []
        fast_sweeps = []                                      # (indices, prepared sweep): same-graph QCMRF lists at release width
        claimed = set()
        if self.sweep_batch and self.width == 'release' and len(circs) > 1:
            from .mrf import QCMRF as _Q
            by_graph = {}
            for i, c in enumerate(circs):
                if type(c) is _Q and not (self.small_batch and c.num_qubits <= small_max):
                    by_graph.setdefault((repr(c._mrf_cliques), c._mrf_measure), []).append(i)
            for idxs in by_graph.values():
                if len(idxs) >= 2:
                    sw = self._qcmrf_release_sweep([circs[i] for i in idxs], n_vars, precision)
                    if sw is not None:
                        fast_sweeps.append((idxs, sw))
                        claimed.update(idxs)
        # Large circuits that run alone are a pipeline: circuit k+1 is prepared and enqueued before circuit k's results
        # are collected (execute_deferred), so the GPU runs the next gate program while the host builds the previous
        # counts dict -- the reference submits its whole list in one run() too (run_experiment.py:56).
        pend = [None]

        def pipeline(item):
            """item = (i, pr, prepare_ms) to enqueue, or None to drain."""
            nxt = None
            if item is not None and pend[0] is not None and (pend[0][1].plan.n_phys != item[1].plan.n_phys or
                                                             pend[0][1].n_vars != item[1].n_vars):
                # another state size replaces the handle, another pmf size the result buffers: finish what is pending
                pipeline(None)
            if item is not None:
                i, pr, tp = item
                te = time.perf_counter()
                fin = self.execute_deferred(pr, shots, seed, sid(i), precision)
                nxt = (i, pr, tp, fin, (time.perf_counter() - te) * 1e3)
            if pend[0] is not None:
                j = pend[0][0]
                entries[j] = self._collect_large(circs[j], *pend[0][1:], sid(j))
            pend[0] = nxt

        for i, c in enumerate(circs):
            if i in claimed:
                continue
            nq = int(c.n_qubits if isinstance(c, ir.Program) else c.num_qubits)
            if self.small_batch and nq <= small_max:
                small_ids.append(i)
                small_prep.append(self.prepare(c, n_vars=n_vars, small=True))
            else:
                tp = time.perf_counter()
                pr = self.prepare(c, n_vars=n_vars)
                tp = (time.perf_counter() - tp) * 1e3
                if self.sweep_batch and len(circs) > 1 and self._sweep_signature(pr, precision) is not None:
                    large.append((i, pr, tp))                 # may join a sweep: decided once every circuit is prepared
                else:
                    pipeline((i, pr, tp))
        pipeline(None)
        # circuits of one program structure (a theta / beta sweep) go through one batched handle
        groups = {}
        if self.sweep_batch and len(large) > 1:
            for k, (i, pr, tp) in enumerate(large):
                sig = self._sweep_signature(pr, precision)
                if sig is not None:
                    groups.setdefault(sig, []).append(k)
        swept = set(k for ks in groups.values() if len(ks) >= 2 for k in ks)
        for k, item in enumerate(large):
            if k not in swept:
                pipeline(item)
        pipeline(None)
        # sweeps last: their post-selected vectors may stay on the GPU, which only holds while the state handle lives
        for idxs, sw in fast_sweeps:
            for e in entries:
                if e is not None and isinstance(e['probs'], _ResidentProbs):
                    e['probs'] = e['probs'].get()
            got = self._run_sweep([circs[i] for i in idxs], None, shots, seed, [sid(i) for i in idxs], precision, pmf, sw=sw)
            for i, e in zip(idxs, got):
                e['name'] = str(getattr(circs[i], 'name', e['name']))
                e['meta']['host_ms'] = {'prepare (vectorised over the sweep)': None}
                entries[i] = e
        for sig, ks in groups.items():
            if len(ks) < 2:
                continue
            for e in entries:                                  # an earlier sweep's resident vectors: bring them home first
                if e is not None and isinstance(e['probs'], _ResidentProbs):
                    e['probs'] = e['probs'].get()
            idxs = [large[k][0] for k in ks]
            got = self._run_sweep([circs[i] for i in idxs], [large[k][1] for k in ks], shots, seed, [sid(i) for i in idxs],
                                  precision, pmf)
            for i, k, e in zip(idxs, ks, got):
                e['meta']['host_ms'] = {'prepare (lower, fuse, plan)': large[k][2]}
                entries[i] = e
        if small_ids:
            ps = [pr.ps if pr.ps is not None else (0, 0, 0) for pr in small_prep]
            keys, probs, kept, ms = _native.run_batch_small(
                [pr.plan for pr in small_prep], [pr.clbit_map for pr in small_prep], ps, shots, seed,
                precision=precision, device=self.device, want_probs=True, stream_ids=[sid(i) for i in small_ids])
            for j, (i, pr) in enumerate(zip(small_ids, small_prep)):
                has_ps = pr.ps is not None
                entries[i] = {
                    'circuit': circs[i], 'name': pr.name,
                    'counts': _keys_to_counts(keys[j], pr.prog.n_clbits) if shots else None,
                    'probs': probs[j].copy() if has_ps else None, 'kept': float(kept[j]) if has_ps else None,
                    'meta': {'path': 'batch_small', 'n_qubits': pr.prog.n_qubits, 'n_phys': pr.plan.n_phys,
                             'passes': pr.plan.n_passes, 'gates_in': pr.fc.n_gates_in, 'batch_device_ms': ms,
                             'philox_stream': sid(i)}}
        res = Result(entries, single, self._name, seed, shots, time.perf_counter() - t0)
        return Job(res)

    # -- sweeps: circuits of one structure through a batched handle ------------------------------------
    def _sweep_signature(self, pr, precision):
        """Hashable program structure of a prepared circuit, or None when it cannot join a batched sweep."""
        pl = pr.plan
        abytes = 8 if precision in ('single', 'c64', 32) else 16
        if (abytes << pl.n_phys) > self.sweep_state_bytes or len(pr.virtual) > 64:
            return None
        if pr.ps is not None and (pr.n_vars > pl.n_phys or not all(pl.layout[q] == q for q in range(pr.n_vars))):
            return None                                       # the post-selected block must be the contiguous stored prefix
        rel = tuple((v['qubit'], tuple(v['ctrl'])) for v in pr.virtual)
        proj = (pr.proj[0].tobytes(), pr.proj[1].size) if pr.proj is not None else None
        return (pl.n_phys, pl.ops.tobytes(), pl.tables.size, pr.clbit_map.tobytes(), pr.ps, rel, proj, pr.prog.n_clbits)

    def prepare_sweep(self, circuits, n_vars=None, precision=None):
        """Prepare a list of same-structure circuits as ONE sweep (raises if their structures differ)."""
        precision = precision or self.precision
        sw = self._qcmrf_release_sweep(list(circuits), n_vars, precision)
        if sw is not None:
            return sw
        prs = [self.prepare(c, n_vars=n_vars) for c in circuits]
        sigs = {self._sweep_signature(pr, precision) for pr in prs}
        if len(sigs) != 1 or None in sigs:
            raise ValueError('prepare_sweep: the circuits do not share one program structure (or their state is too large '
                             'for a batched sweep: sweep_state_bytes)')
        return self._stack_sweep(prs)

    def _qcmrf_release_sweep(self, circs, n_vars, precision):
        """A theta / beta sweep of pristine QCMRF objects over ONE graph at release width, prepared in one
        vectorised pass: the first circuit is prepared in full; for the others only the coefficients change, and
        at release width every one of them is an elementwise function of gamma (P(ancilla = 1 | x_C) = sin^2 2gamma,
        projection factors = merged products of cos 2gamma) -- computed here for all points at once instead of
        lowering, fusing and planning 256 circuits.  Returns None whenever the shortcut does not apply."""
        from .mrf import QCMRF
        if self.width != 'release' or len(circs) < 2:
            return None
        c0 = circs[0]
        for c in circs:
            if (type(c) is not QCMRF or c.__dict__.get('_mrf_data') is not None or c._mrf_measure != c0._mrf_measure
                    or c._mrf_cliques != c0._mrf_cliques):
                return None
        pr0 = self.prepare(c0, n_vars=n_vars)
        if (not pr0.virtual or pr0.fc.ops or pr0.proj is None or self._sweep_signature(pr0, precision) is None
                or len(pr0.virtual) != len(c0._mrf_cliques)):
            return None                                   # not every clique sweep is released: general path
        st = c0.__dict__.get('_mrf_struct')
        if not st:
            return None
        B, dim = len(circs), c0._mrf_dim
        G = np.empty((B, dim))
        with np.errstate(invalid='ignore'):
            for y, c in enumerate(circs):
                if c._mrf_gamma is not None:
                    G[y] = c._mrf_gamma
                else:
                    G[y] = 0.5 * np.arccos(np.exp(c._mrf_beta * 0.5 * np.asarray(c._mrf_theta, dtype=np.float64)))
        if not np.isfinite(G).all():
            raise ValueError('QCMRF: theta must be <= 0 (gamma is not finite)')
        if not (np.abs(G) > 1e-8).all():
            return None                                   # skipped terms (QCMRF.py:223) change the structure: general path
        cosg, sing = np.cos(2.0 * G), np.sin(2.0 * G)
        gidx = {}
        for m, ids, idx in st:
            for r, ii in enumerate(ids):
                gidx[ii] = idx[r]
        pl = pr0.plan
        n = c0._mrf_n
        diag, p1 = [], []
        for v in pr0.virtual:                             # released sweeps, in program order: clique ii's ancilla is qubit n+1+ii
            ii = v['qubit'] - n - 1
            a0, a1 = cosg[:, gidx[ii]], sing[:, gidx[ii]]
            w0, w1 = a0 * a0, a1 * a1
            p1.append(w1 / (w0 + w1))
            diag.append((v['ctrl'], a0))
        steps = fusion._merge_steps(tuple(tuple(int(c) for c in ctrl) for ctrl, _d in diag))
        merged, cur_ctrl, cur = [], [], np.ones((B, 1))
        for (flush, union, ia, ib), (_ctrl, d) in zip(steps, diag):
            if flush:
                merged.append((cur_ctrl, cur))
                cur = np.ones((B, 1))
            cur = cur[:, ia] * d[:, ib]
            cur_ctrl = list(union)
        merged.append((cur_ctrl, cur))
        merged = [fusion.sort_diag_ctrl(c, t) for c, t in merged]
        proj_ops, proj_t0 = pr0.proj
        dops = [o for o in proj_ops if int(o['kind']) == fusion.QCM_OP_DIAG]
        if len(dops) != len(merged) or any(list(o['ctrl'][:int(o['n_ctrl'])]) != list(c) for o, (c, _t) in zip(dops, merged)):
            return None
        proj_tables = np.zeros((B, proj_t0.size))
        for o, (_c, t) in zip(dops, merged):
            off = int(o['table_off'])
            proj_tables[:, off:off + 2 * t.shape[1]:2] = t          # real parts; the factors are real (cos 2 gamma)
        sw = _Sweep()
        sw.prs = [pr0] * B
        sw.ops, sw.n_phys, sw.ps, sw.clbit_map, sw.n_vars = pl.ops, pl.n_phys, pr0.ps, pr0.clbit_map, pr0.n_vars
        sw.tables = np.broadcast_to(pl.tables, (B, pl.tables.size))  # the stored qubits' program (H layer) has no theta in it
        sw.proj_ops, sw.proj_tables = proj_ops, proj_tables
        sw.released = self._released_tables(pr0)
        sw.p1 = np.ascontiguousarray(np.concatenate(p1, axis=1))
        return sw

    def _stack_sweep(self, prs):
        sw = _Sweep()
        p0 = prs[0]
        sw.prs, sw.ops, sw.n_phys, sw.ps, sw.clbit_map, sw.n_vars = prs, p0.plan.ops, p0.plan.n_phys, p0.ps, p0.clbit_map, p0.n_vars
        sw.tables = np.stack([pr.plan.tables for pr in prs])
        sw.proj_ops = sw.proj_tables = sw.released = sw.p1 = None
        if p0.virtual:
            sw.proj_ops = p0.proj[0]
            sw.proj_tables = np.stack([pr.proj[1] for pr in prs])
            sw.released = self._released_tables(p0)
            sw.p1 = np.stack([self._released_tables(pr)[3] for pr in prs])
        return sw

    def execute_sweep(self, sw, shots, seed=0, streams=None, precision=None, pmf=None, first=0, count=None, profile=False):
        """Run points [first, first + count) of a prepared sweep through one batched handle: program, shots (released
        qubits drawn on the device), projection + post-selection.  Returns (keys (count, shots) or None, probs --
        (count, 2^n) array if pmf is True, a list of _ResidentProbs if pmf is None, else None --, kept (count,) or None).
        The calls are enqueued in the engine's deferred mode (one synchronisation at the end, results into page-locked
        buffers that are reused by the next sweep of the same shape); profile=True runs them one by one instead and
        leaves the per-launch record in `sweep_profile`."""
        precision = precision or self.precision
        B = len(sw.prs) - first if count is None else count
        sl = slice(first, first + B)
        if streams is None:
            streams = np.arange(first, first + B, dtype=np.uint64)
        if B == 1:
            raise ValueError('a sweep chunk needs at least two points')
        h = self._handle(sw.n_phys, precision, batch=B)
        self._last = h
        deferred = not profile and hasattr(h, 'set_deferred')
        keys_out = kept_out = None
        if deferred:
            pin = self._pinned.get((B, shots))
            if pin is None:
                self._pinned.clear()
                pin = self._pinned[(B, shots)] = (_native.PinnedArray((B, max(shots, 1)), np.uint64), _native.PinnedArray((B,), np.float64))
            keys_out, kept_out = pin[0].array, pin[1].array
            h.set_deferred(True)
        try:
            tw = [time.perf_counter()]
            h.run_program(sw.ops, sw.tables[sl])
            tw.append(time.perf_counter())
            prof = {'program': [] if deferred else list(zip(h.op_kernels(), h.op_profile())), 'projection': [], 'points': B}
            keys = None
            if shots:
                if sw.released is not None:
                    mc, n_ctrl, ctrl, _p1, p1_off, vclbit, clbit_pos, n_cl = sw.released
                    keys = h.sample_released_batched(shots, seed, streams, n_ctrl, ctrl, sw.p1[sl], p1_off, vclbit, clbit_pos, n_cl,
                                                     **({'out': keys_out} if deferred else {}))
                else:
                    keys = h.sample_batched(shots, seed, streams, sw.clbit_map if len(sw.clbit_map) else None,
                                            **({'out': keys_out} if deferred else {}))
            tw.append(time.perf_counter())
            probs = kept = None
            if pmf is not False and sw.ps is not None and sw.n_vars <= 30:
                if sw.proj_ops is not None:
                    h.run_program(sw.proj_ops, sw.proj_tables[sl])      # project the released qubits on 0 (after the shots)
                    if not deferred:
                        prof['projection'] = list(zip(h.op_kernels(), h.op_profile()))
                tw.append(time.perf_counter())
                mask, value, n = sw.ps
                if pmf:
                    if deferred:                                  # the full vectors come to pageable memory: finish what is queued first
                        h.synchronize()
                        h.set_deferred(False)
                    probs, kept = h.postselect(mask, value, n)
                else:
                    kept = h.postselect_resident(mask, value, n, **({'out': kept_out} if deferred else {}))
                    probs = [_ResidentProbs(h, y, n) for y in range(B)]
            if deferred:
                h.synchronize()
        finally:
            if deferred:
                h.set_deferred(False)
        tw.append(time.perf_counter())
        t = h.timing()
        prof['sample_ms'], prof['postselect_ms'] = (t['sample_ms'] if shots else 0.0), (t['postselect_ms'] if kept is not None else 0.0)
        prof['host_wall_ms'] = [round((b - a) * 1e3, 3) for a, b in zip(tw[:-1], tw[1:])]   # program, shots, projection, post-selection
        prof['deferred'] = bool(deferred)
        self.sweep_profile = prof                             # record of the last sweep chunk (bench.py)
        return keys, probs, kept

    def _run_sweep(self, circs, prs, shots, seed, streams, precision, pmf, sw=None):
        if sw is None:
            sw = self._stack_sweep(prs)
        prs = sw.prs
        abytes = 8 if precision in ('single', 'c64', 32) else 16
        # points per batched handle: sweep_bytes of state, and never more than the engine takes (qcm_create_batched)
        cap = min(SWEEP_MAX_POINTS, max(2, int(self.sweep_bytes // (abytes << sw.n_phys))))
        entries = []
        n = len(prs)
        first = 0
        while first < n:
            B = min(cap, n - first)
            if n - first - B == 1:                            # never leave a chunk of one point
                B -= 1
            if B < 2:                                         # (n - first == 1 cannot happen: chunks are >= 2)
                B = n - first
            t0 = time.perf_counter()
            # a later chunk reuses the handle: resident vectors of the earlier chunk must come to the host first
            for e in entries:
                if isinstance(e['probs'], _ResidentProbs):
                    e['probs'] = e['probs'].get()
            keys, probs, kept = self.execute_sweep(sw, shots, seed, np.asarray(streams[first:first + B], dtype=np.uint64), precision,
                                                   pmf, first, B)
            t1 = time.perf_counter()
            h = self._last
            t = h.timing()
            for y in range(B):
                pr = prs[first + y]
                counts = _keys_to_counts(keys[y], pr.prog.n_clbits) if shots else None
                pv = None if probs is None else probs[y]
                entries.append({'circuit': circs[first + y], 'name': pr.name, 'counts': counts, 'probs': pv,
                                'kept': None if kept is None else float(kept[y]),
                                'meta': {'path': 'sweep', 'width': 'release' if pr.virtual else 'full', 'sweep_points': B,
                                         'released_qubits': len(pr.virtual), 'n_qubits': pr.prog.n_qubits, 'n_phys': sw.n_phys,
                                         'passes': pr.plan.n_passes, 'gates_in': pr.fc.n_gates_in, 'philox_stream': int(streams[first + y]),
                                         'h2d_bytes': int(sw.tables[0].nbytes + sw.ops.nbytes + (sw.proj_tables[0].nbytes if sw.proj_tables is not None else 0)
                                                          + (sw.p1[0].nbytes if sw.p1 is not None else 0)),
                                         'd2h_bytes': int((keys[y].nbytes if keys is not None else 0) + 8
                                                          + (probs[y].nbytes if isinstance(probs, np.ndarray) else 0)),
                                         'sweep_execute_ms': (t1 - t0) * 1e3, 'sample_ms': t['sample_ms'],
                                         'postselect_ms': t['postselect_ms']}})
            first += B
        return entries

    def execute(self, pr, shots, seed=0, stream=0, precision=None, want_probs=True):
        """Run one prepared circuit on the large-state path: program, post-selection, shots.
        Returns (keys or None, probs or None, kept or None)."""
        pl = pr.plan
        h = self._handle(pl.n_phys, precision or self.precision)
        self._last = h
        ops = pl.ops
        if (not shots or pr.virtual) and len(ops) and ops['flags'].any():
            ops = ops.copy()
            if pr.virtual:
                ops['flags'] = 0               # projection passes follow on the same state: plain layout, no checkpoint
            else:
                ops['flags'] &= ~fusion.QCM_FLAG_SAMPLE_CHECKPOINT     # no shots follow: skip the sampler's checkpoint tree
        h.run_program(ops, pl.tables)
        keys = None
        if shots and pr.virtual:
            keys = self._sample_released(h, pr, shots, seed, stream)
        elif shots:
            keys = h.sample(shots, seed, stream, pr.clbit_map if len(pr.clbit_map) else None)
        probs = kept = None
        if want_probs and pr.ps is not None and pr.n_vars <= 30:
            if pr.virtual:
                h.run_program(*pr.proj)        # project the released qubits on 0 (after the shots were drawn)
            probs, kept = self._probs_from_handle(h, pr)
        return keys, probs, kept

    def execute_deferred(self, pr, shots, seed=0, stream=0, precision=None):
        """ENQUEUE one prepared circuit on the large-state path -- program, shots, post-selection, all into page-locked
        result buffers (a ring of three) -- and return a zero-argument callable that waits for THIS circuit's results
        (qcm_mark / qcm_wait) and returns what execute() returns.  Between the two calls the next circuit can be prepared
        and enqueued: a list of circuits then runs back to back on the GPU while the host formats the previous result
        (run() does exactly that).  Same kernels, same Philox streams, same results as execute().  Falls back to the
        blocking execute() where the pipeline does not apply (release width, no shots, variables off the low qubits)."""
        pl = pr.plan
        precision = precision or self.precision
        h = self._handle(pl.n_phys, precision)
        n = pr.n_vars
        if not (shots and not pr.virtual and pr.ps is not None and n is not None and n <= min(30, pl.n_phys) and hasattr(h, 'mark')
                and all(pl.layout[q] == q for q in range(n))):
            out = self.execute(pr, shots, seed, stream, precision)
            return lambda: out
        self._last = h
        key = (1 << n, int(shots))
        ring = self._ring
        if ring is None or ring['key'] != key:
            if ring is not None:
                for rec in ring['busy']:
                    if rec is not None and not rec['done']:
                        raise RuntimeError('deferred executions of another shape are still pending: finish them first')
            ring = self._ring = {'key': key, 'slot': 0, 'busy': [None] * 3,
                                 'bufs': [(_native.PinnedArray((int(shots),), np.uint64), _native.PinnedArray((1 << n,), np.float64),
                                           _native.PinnedArray((1,), np.float64)) for _ in range(3)]}
        slot = ring['slot']
        ring['slot'] = (slot + 1) % 3
        old = ring['busy'][slot]
        if old is not None and not old['done']:
            raise RuntimeError('deferred executions must be finished (call what execute_deferred returned) before three '
                               'more are started')
        kb, pb, mb = ring['bufs'][slot]
        mask, value, _ = pr.ps
        h.set_deferred(True)
        try:
            h.run_program(pl.ops, pl.tables)
            h.sample(shots, seed, stream, pr.clbit_map if len(pr.clbit_map) else None, out=kb.array)
            h.postselect(mask, value, n, out=(pb.array, mb.array))
            ticket = h.mark()
        finally:
            h.set_deferred(False)
        rec = {'done': False}
        ring['busy'][slot] = rec

        def finish():
            if rec['done']:
                raise RuntimeError('this deferred execution was already collected')
            h.wait(ticket)
            out = (kb.array.copy(), pb.array.copy(), float(mb.array[0]))
            rec['done'] = True                            # the slot's page-locked buffers may be reused
            return out
        finish.deferred = True
        return finish

    def _sample_released(self, h, pr, shots, seed, stream):
        """Shots of a circuit whose released qubits are not stored: basis states of the stored qubits
        come from the GPU sampler, each released qubit's outcome from its sweep's coefficients at that
        basis state.  On the GPU engine that second step runs on the device too (qcm_sample_released); the
        host version below (numpy Philox keyed by (seed, stream), one column per released qubit) serves an
        engine without that entry point (the tests' numpy stand-in)."""
        pl = pr.plan
        if hasattr(h, 'sample_released') and len(pr.virtual) <= 64:
            # the engine draws the released qubits itself (k_released_keys, device Philox): one call, one read-back
            mc, n_ctrl, ctrl, p1, p1_off, vclbit, clbit_pos, n_cl = self._released_tables(pr)
            return h.sample_released(shots, seed, stream, n_ctrl, ctrl, p1, p1_off, vclbit, clbit_pos, n_cl)
        raw = h.sample(shots, seed, stream, None).astype(np.int64)
        rng = np.random.Generator(np.random.Philox(key=[int(seed) & (2 ** 64 - 1), int(stream) & (2 ** 64 - 1)]))
        u = rng.random((len(pr.virtual), shots))
        L = _host()
        if L:
            return self._released_keys_native(L, pr, raw, u)
        vbits = {}
        for k, v in enumerate(pr.virtual):
            idx = np.zeros(shots, dtype=np.int64)
            for j, c in enumerate(v['ctrl']):
                idx |= ((raw >> c) & 1) << j
            vbits[v['qubit']] = (u[k] < v['p1'][idx]).astype(np.uint64)
        keys = np.zeros(shots, dtype=np.uint64)
        for c, q in pr.prog.measures.items():
            if q in vbits:
                keys |= vbits[q] << np.uint64(c)
            elif pl.layout[q] < pl.n_phys:
                keys |= ((raw >> pl.layout[q]) & 1).astype(np.uint64) << np.uint64(c)
        return keys

    @staticmethod
    def _released_tables(pr):
        """Flat arrays describing the released qubits of a prepared circuit (cached on it)."""
        pl = pr.plan
        nv = len(pr.virtual)
        tabs = getattr(pr, '_released_tabs', None)
        if tabs is None:
            mc = max([len(v['ctrl']) for v in pr.virtual] + [1])
            n_ctrl = np.array([len(v['ctrl']) for v in pr.virtual], dtype=np.int32)
            ctrl = np.zeros((nv, mc), dtype=np.int32)
            for k, v in enumerate(pr.virtual):
                ctrl[k, :len(v['ctrl'])] = v['ctrl']
            p1 = np.ascontiguousarray(np.concatenate([np.asarray(v['p1'], dtype=np.float64) for v in pr.virtual]))
            p1_off = np.concatenate([[0], np.cumsum([len(v['p1']) for v in pr.virtual])[:-1]]).astype(np.int64)
            vq = {v['qubit']: k for k, v in enumerate(pr.virtual)}
            vclbit = np.full(nv, -1, dtype=np.int32)
            n_cl = (max(pr.prog.measures) + 1) if pr.prog.measures else 0
            clbit_pos = np.full(max(n_cl, 1), -1, dtype=np.int32)
            for c, q in pr.prog.measures.items():
                if q in vq:
                    vclbit[vq[q]] = c
                elif pl.layout[q] < pl.n_phys:
                    clbit_pos[c] = pl.layout[q]
            tabs = pr._released_tabs = (mc, n_ctrl, ctrl, p1, p1_off, vclbit, clbit_pos, n_cl)
        return tabs

    @classmethod
    def _released_keys_native(cls, L, pr, raw, u):
        """The host-side key assembly in one pass over the shots (csrc/qcm_host.c, qcm_released_keys)."""
        nv, shots = len(pr.virtual), len(raw)
        mc, n_ctrl, ctrl, p1, p1_off, vclbit, clbit_pos, n_cl = cls._released_tables(pr)
        raw = np.ascontiguousarray(raw, dtype=np.int64)
        u = np.ascontiguousarray(u, dtype=np.float64)
        keys = np.empty(shots, dtype=np.uint64)
        rc = L.qcm_released_keys(raw.ctypes.data, shots, u.ctypes.data, nv, n_ctrl.ctypes.data, ctrl.ctypes.data, mc,
                                 p1.ctypes.data, p1_off.ctypes.data, vclbit.ctypes.data, clbit_pos.ctypes.data, n_cl,
                                 keys.ctypes.data)
        if rc:
            raise ValueError('qcm_released_keys: bad arguments')
        return keys

    def kernel_launches(self):
        """Kernels launched so far by the live state handles (bench.py's gpu_launches)."""
        return self._launches_closed + sum(h.timing()['kernel_launches'] for h in self._handles.values())

    def last_timing(self):
        return self._last.timing() if self._last is not None else None

    def op_profile(self):
        """Per-launch (kind, ms, bytes_read, bytes_written) of the last executed program."""
        return self._last.op_profile()

    def op_kernels(self):
        """Kernel name per entry of op_profile() ('' where the engine does not record one)."""
        return self._last.op_kernels()

    def _collect_large(self, circ, pr, prepare_ms, finish, enqueue_ms, stream):
        """Entry of one large-state circuit from its pending execution (see run())."""
        pl = pr.plan
        t0 = time.perf_counter()
        keys, probs, kept = finish()
        t1 = time.perf_counter()
        h = self._last
        shots = 0 if keys is None else len(keys)
        counts = _keys_to_counts(keys, pr.prog.n_clbits) if shots else None
        pmf = _normalised(probs, kept)
        t2 = time.perf_counter()
        t = h.timing()
        if getattr(finish, 'deferred', False):                # enqueued executions collect no per-phase device timings
            t = dict(t, program_ms=None, sample_ms=None, postselect_ms=None)
        self.breakdown_ms = {'prepare (lower, fuse, plan)': prepare_ms, 'execute or enqueue (program, shots, post-selection)': enqueue_ms,
                             'wait for the results': (t1 - t0) * 1e3, 'counts dict': (t2 - t1) * 1e3}
        h2d = pl.ops.nbytes + pl.tables.nbytes + (pr.clbit_map.nbytes if shots else 0)
        d2h = (probs.nbytes + 8 if probs is not None else 0) + (keys.nbytes if keys is not None else 0)
        return {'circuit': circ, 'name': pr.name, 'counts': counts, 'probs': None if pmf is not None else probs, 'pmf': pmf, 'kept': kept,
                'meta': {'path': 'statevector', 'width': 'release' if pr.virtual else 'full',
                         'released_qubits': len(pr.virtual), 'n_qubits': pr.prog.n_qubits, 'n_phys': pl.n_phys,
                         'passes': pl.n_passes, 'gates_in': pr.fc.n_gates_in, 'program_ms': t['program_ms'],
                         'sample_ms': t['sample_ms'], 'postselect_ms': t['postselect_ms'],
                         'bytes_read': t['bytes_read'], 'bytes_written': t['bytes_written'],
                         'h2d_bytes': int(h2d), 'd2h_bytes': int(d2h), 'philox_stream': stream,
                         'host_ms': dict(self.breakdown_ms)}}

    def exact(self, circuit, n=None, precision=None):
        """Exact post-selected probability vector and success probability (no shots)."""
        res = self.run(circuit, shots=0, n_vars=n, precision=precision).result()
        return res.postselected_probabilities(0)

    def statevector(self, circuit, precision=None):
        """Full logical statevector (small circuits; for tests and debugging)."""
        precision = precision or self.precision
        pr = self.prepare(circuit, fusion_mode=self.fusion)
        pl = pr.plan
        if pl.n_logical > 26:
            raise ValueError('statevector() is meant for small circuits')
        h = self._handle(pl.n_phys, precision)
        h.run_program(pl.ops, pl.tables)
        phys = h.get_amplitudes(0, 1 << pl.n_phys).astype(np.complex128)
        N = pl.n_logical
        idx = np.arange(1 << N)
        pidx = np.zeros(1 << N, dtype=np.int64)
        dead = np.zeros(1 << N, dtype=bool)
        for q in range(N):
            b = (idx >> q) & 1
            if pl.layout[q] < pl.n_phys:
                pidx |= b << pl.layout[q]
            else:
                dead |= b == 1
        out = phys[pidx]
        out[dead] = 0.0
        return out * np.exp(1j * pl.global_phase)
