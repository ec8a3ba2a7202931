"""CPU stand-in for the CUDA engine, for HOST-LOGIC tests only.

TEST INFRASTRUCTURE: executes engine programs with tests/engine_emulator.py (numpy)
so that the lowering / fusion / planning / key-formatting code -- and the
reference's own scripts on top of it -- can be exercised in the GPU-less build
container.  It is monkeypatched over qcmrf_b200._native by the tests that need it;
the product has no such path (without the CUDA library it raises).
"""
import numpy as np

import engine_emulator as em


class FakePlanHolder:
    pass


def _keys_from_probs(p, shots, rng, clbit_map):
    idx = rng.choice(len(p), size=shots, p=p / p.sum())
    if clbit_map is None or len(clbit_map) == 0:
        return idx.astype(np.uint64)
    keys = np.zeros(shots, dtype=np.uint64)
    for c, q in enumerate(clbit_map):
        if q >= 0:
            keys |= ((idx >> int(q)) & 1).astype(np.uint64) << np.uint64(c)
    return keys


def small_max_qubits(precision='double'):
    return 13


def run_batch_small(plans, clbit_maps, ps, shots, seed, precision='double', device=0, want_probs=True,
                    stream_ids=None):
    n = len(plans)
    keys = np.zeros((n, shots), dtype=np.uint64) if shots else None
    probs, kept = [], np.zeros(n)
    for i, pl in enumerate(plans):
        phys, act = em.run_plan(pl)
        w = np.abs(phys) ** 2
        mask, value, bits = ps[i]
        idx = np.arange(len(w))
        sel = (idx & mask) == value
        out = np.zeros(1 << bits)
        np.add.at(out, idx[sel] & ((1 << bits) - 1), w[sel])
        probs.append(out)
        kept[i] = w[sel].sum()
        if shots:
            sid = i if stream_ids is None else int(stream_ids[i])
            rng = np.random.default_rng([seed & 0xffffffff, sid])
            keys[i] = _keys_from_probs(w, shots, rng, clbit_maps[i])
    return keys, probs, kept, 0.0


class Handle:
    """numpy stand-in for _native.Handle.  With ``ext_state_ptr`` the state aliases caller memory
    (a torch CPU tensor in the gloo tests), as the real handle aliases a torch CUDA tensor."""

    def __new__(cls, n_local, precision='single', device=0, ext_state_ptr=None, ext_stream=None, batch=1):
        if batch > 1 and cls is Handle:
            return object.__new__(BatchedHandle)
        return object.__new__(cls)

    def __init__(self, n_local, precision='single', device=0, ext_state_ptr=None, ext_stream=None, batch=1):
        import ctypes
        self.batch = 1
        self.generation = 0
        self._h = True
        self.n_local = n_local
        self.cdtype = np.complex64 if precision in ('single', 'c64', 32) else np.complex128
        self.ext = None
        if ext_state_ptr:
            rt = ctypes.c_float if self.cdtype == np.complex64 else ctypes.c_double
            buf = (rt * (2 << n_local)).from_address(ext_state_ptr)
            self.ext = np.ctypeslib.as_array(buf).view(self.cdtype)
        self._own = np.zeros(1 << n_local, dtype=np.complex128)
        self.active = 0
        self.n_global = 0
        self.rank = 0
        self._prof = []

    @property
    def state(self):
        return self.ext.astype(np.complex128) if self.ext is not None else self._own

    def _store(self, psi):
        psi = np.where(np.isnan(psi), 0, psi)
        if self.ext is not None:
            self.ext[:] = psi.astype(self.cdtype)
        else:
            self._own = psi

    def set_shard(self, n_global, rank):
        self.n_global, self.rank = n_global, rank

    def run_program(self, ops, tables):
        pl = FakePlanHolder()
        pl.ops, pl.tables, pl.n_phys = ops, tables, self.n_local
        # a state of ZERO active qubits (one amplitude: every local qubit still unmaterialised) is a state too
        psi0 = self.state if getattr(self, '_has_state', False) else None
        psi, self.active = em.run_plan(pl, n_global=self.n_global, rank=self.rank, n_local=self.n_local,
                                       psi0=psi0, active0=self.active if psi0 is not None else 0)
        self._store(psi)
        self._has_state = True
        self._prof = [(int(o['kind']), 0.0, 0, 0) for o in ops]

    def _global_index(self):
        return np.arange(1 << self.n_local, dtype=np.int64) | (self.rank << self.n_local)

    def postselect(self, mask, value, n_out_bits, want_probs=True, out=None):
        if not 0 <= n_out_bits <= min(self.n_local, 30):
            raise RuntimeError('n_out_bits %d out of range' % n_out_bits)        # as qcm_postselect refuses it
        w = np.abs(self.state) ** 2
        w[1 << self.active:] = 0
        idx = self._global_index()
        sel = (idx & mask) == value
        res = np.zeros(1 << n_out_bits)
        np.add.at(res, idx[sel] & ((1 << n_out_bits) - 1), w[sel])
        if out is not None:                                 # deferred mode of the real handle: caller-owned buffers
            out[0][:] = res
            out[1][0] = float(w[sel].sum())
            return out
        return res, float(w[sel].sum())

    def sample(self, shots, seed, stream_id=0, clbit_qubit=None, out=None):
        rng = np.random.default_rng([seed & 0xffffffff, stream_id])
        keys = _keys_from_probs(np.abs(self.state) ** 2, shots, rng, clbit_qubit)
        if out is not None:
            out[:] = keys
            return out
        return keys

    # the real handle enqueues in deferred mode and waits per ticket; the emulator runs everything at once, so the
    # host-side pipeline (ring slots, collection order) is what these exercise
    def set_deferred(self, flag):
        self.deferred = bool(flag)

    def mark(self):
        self._tickets = getattr(self, '_tickets', 0) + 1
        return self._tickets - 1

    def wait(self, ticket):
        if ticket >= getattr(self, '_tickets', 0):
            raise RuntimeError('ticket %d was never issued' % ticket)

    def sample_prepare(self):
        w = np.abs(self.state) ** 2
        w[1 << self.active:] = 0
        return float(w.sum())

    def sample_sharded(self, shots, seed, stream_id, rank_masses, clbit_qubit=None):
        """Every rank draws the same uniforms; a shot belongs to the rank whose mass interval holds it."""
        rng = np.random.default_rng([seed & 0xffffffff, stream_id])
        u = rng.random(shots) * float(np.sum(rank_masses))
        edges = np.concatenate([[0.0], np.cumsum(rank_masses)])
        lo, hi = edges[self.rank], edges[self.rank + 1]
        if self.rank == len(rank_masses) - 1:
            hi = np.inf
        mine = (u >= lo) & (u < hi)
        w = np.abs(self.state) ** 2
        w[1 << self.active:] = 0
        cdf = np.cumsum(w)
        loc = np.searchsorted(cdf, np.clip(u - lo, 0, cdf[-1] * (1 - 1e-15)), side='right')
        loc = np.minimum(loc, len(w) - 1)
        gi = loc.astype(np.int64) | (self.rank << self.n_local)
        keys = np.zeros(shots, dtype=np.uint64)
        if clbit_qubit is None or len(clbit_qubit) == 0:
            keys = gi.astype(np.uint64)
        else:
            for c, q in enumerate(clbit_qubit):
                if q >= 0:
                    keys |= ((gi >> int(q)) & 1).astype(np.uint64) << np.uint64(c)
        keys[~mine] = 0
        return keys, mine

    def get_amplitudes(self, first=0, count=None):
        st = self.state
        count = len(st) - first if count is None else count
        return st[first:first + count].astype(self.cdtype)

    def get_active(self):
        return self.active

    def op_profile(self):
        return list(self._prof)

    def op_kernels(self):
        return [''] * len(self._prof)

    def timing(self):
        return dict(program_ms=0.0, sample_ms=0.0, postselect_ms=0.0, kernel_launches=0, bytes_read=0,
                    bytes_written=0)

    def close(self):
        self._h = None


class BatchedHandle(Handle):
    """numpy stand-in for a batched handle (qcm_create_batched): `batch` independent states, shared ops,
    per-point tables as rows."""

    def __init__(self, n_local, precision='single', device=0, ext_state_ptr=None, ext_stream=None, batch=1):
        self.batch = batch
        self.generation = 0
        self._h = True
        self.n_local = n_local
        self.pts = [Handle(n_local, precision) for _ in range(batch)]
        self._resident = None

    def run_program(self, ops, tables):
        tables = np.asarray(tables)
        assert tables.ndim == 2 and tables.shape[0] == self.batch
        for h, t in zip(self.pts, tables):
            h.run_program(ops, t)

    def postselect(self, mask, value, n_out_bits, want_probs=True):
        self.generation += 1
        got = [h.postselect(mask, value, n_out_bits) for h in self.pts]
        return (np.stack([g[0] for g in got]) if want_probs else None), np.array([g[1] for g in got])

    def postselect_resident(self, mask, value, n_out_bits, out=None):
        probs, kept = self.postselect(mask, value, n_out_bits)
        self._resident = probs
        if out is not None:
            out[:] = kept
            return out
        return kept

    def synchronize(self):
        pass

    def fetch_probs(self, point, n_out_bits, first=0, count=None):
        return self._resident[point][first:None if count is None else first + count].copy()

    def sample_batched(self, shots, seed, stream_ids, clbit_qubit=None, out=None):
        keys = np.stack([h.sample(shots, seed, int(sid), clbit_qubit) for h, sid in zip(self.pts, stream_ids)])
        if out is not None:
            out[:] = keys
            return out
        return keys

    def sample_released_batched(self, shots, seed, stream_ids, n_ctrl, ctrl, p1, p1_off, vclbit, clbit_pos, n_clbits, out=None):
        out = np.zeros((self.batch, shots), dtype=np.uint64) if out is None else out
        for y, (h, sid) in enumerate(zip(self.pts, stream_ids)):
            raw = h.sample(shots, seed, int(sid), None).astype(np.int64)
            rng = np.random.default_rng([seed & 0xffffffff, int(sid), 7])
            keys = np.zeros(shots, dtype=np.uint64)
            for c in range(n_clbits):
                if clbit_pos[c] >= 0:
                    keys |= ((raw >> int(clbit_pos[c])) & 1).astype(np.uint64) << np.uint64(c)
            for k in range(len(n_ctrl)):
                if vclbit[k] < 0:
                    continue
                idx = np.zeros(shots, dtype=np.int64)
                for j in range(int(n_ctrl[k])):
                    idx |= ((raw >> int(ctrl[k, j])) & 1) << j
                bit = rng.random(shots) < p1[y][int(p1_off[k]) + idx]
                keys |= bit.astype(np.uint64) << np.uint64(int(vclbit[k]))
            out[y] = keys
        return out

    def op_profile(self):
        return self.pts[0].op_profile()

    def op_kernels(self):
        return self.pts[0].op_kernels()

    def timing(self):
        return dict(program_ms=0.0, sample_ms=0.0, postselect_ms=0.0, kernel_launches=0, bytes_read=0, bytes_written=0)

    def close(self):
        self._h = None


class PinnedArray:
    """numpy stand-in for _native.PinnedArray (page-locked host memory)."""

    def __init__(self, shape, dtype):
        self.array = np.zeros(shape, dtype=dtype)


def install(monkeypatch):
    from qcmrf_b200 import _native
    monkeypatch.setattr(_native, 'PinnedArray', PinnedArray)
    monkeypatch.setattr(_native, 'small_max_qubits', small_max_qubits)
    monkeypatch.setattr(_native, 'run_batch_small', run_batch_small)
    monkeypatch.setattr(_native, 'Handle', Handle)
