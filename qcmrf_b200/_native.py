"""ctypes binding of the C ABI declared in include/qcmrf_b200.h.

There is deliberately no fallback: if the shared library is missing, or the
machine has no CUDA device, every compute call raises.
"""
import ctypes
import os

import numpy as np

from .fusion import OP_DTYPE

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libqcmrf_b200.so')

QCM_C64, QCM_C128 = 32, 64
_STATUS = {0: 'QCM_OK', -1: 'QCM_ERR_INVALID', -2: 'QCM_ERR_CUDA', -3: 'QCM_ERR_NOMEM',
           -4: 'QCM_ERR_UNSUPPORTED', -5: 'QCM_ERR_NO_DEVICE'}


class NativeError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__('%s (%d): %s' % (_STATUS.get(code, '?'), code, msg))
        self.code = code


class QcmTiming(ctypes.Structure):
    _fields_ = [('program_ms', ctypes.c_double), ('sample_ms', ctypes.c_double),
                ('postselect_ms', ctypes.c_double), ('kernel_launches', ctypes.c_uint64),
                ('bytes_read', ctypes.c_uint64), ('bytes_written', ctypes.c_uint64)]


_lib = None

# every symbol include/qcmrf_b200.h declares (tests check the .so exports all of them)
SYMBOLS = ['qcm_abi_version', 'qcm_device_count', 'qcm_last_error', 'qcm_create', 'qcm_destroy',
           'qcm_set_shard', 'qcm_get_amplitudes', 'qcm_set_amplitudes', 'qcm_synchronize',
           'qcm_run_program', 'qcm_postselect', 'qcm_sample', 'qcm_sample_prepare', 'qcm_sample_sharded',
           'qcm_small_max_qubits', 'qcm_run_batch_small', 'qcm_state_ptr', 'qcm_set_active',
           'qcm_get_active', 'qcm_get_timing', 'qcm_get_op_profile', 'qcm_postselect_device',
           'qcm_sample_sharded_device', 'qcm_run_gather_block', 'qcm_enable_peer_access',
           'qcm_ipc_export', 'qcm_ipc_open', 'qcm_ipc_close', 'qcm_op_kernel_name',
           'qcm_sample_released', 'qcm_create_batched', 'qcm_batch_size', 'qcm_batch_select',
           'qcm_postselect_resident', 'qcm_fetch_probs', 'qcm_sample_batched', 'qcm_sample_released_batched',
           'qcm_sample_sharded_devmass', 'qcm_mrf_exact', 'qcm_mrf_last_error', 'qcm_gather_flag_words',
           'qcm_run_gather_block_inplace', 'qcm_set_deferred', 'qcm_host_alloc', 'qcm_host_free',
           'qcm_tree_total_device', 'qcm_mark', 'qcm_wait', 'qcm_run_batch_small_readout', 'qcm_run_noisy_small', 'qcm_tree_level',
           'qcm_run_noisy_small_kraus']

#: qcm_gate and qcm_channel of include/qcmrf_b200.h (the noisy-shot launch)
GATE_DTYPE = np.dtype([('m', '<f8', (8,)), ('target', '<i4'), ('ctrl_mask', '<u4'), ('ctrl_value', '<u4'),
                       ('channel', '<i4')])
CHANNEL_DTYPE = np.dtype([('cum', '<f8', (16,)), ('n_paulis', '<i4'), ('qubit', '<i4', (2,)), ('pad', '<i4')])
#: qcm_gate_error and qcm_kraus (qcm_run_noisy_small_kraus)
GATE_ERROR_DTYPE = np.dtype([('n_stages', '<i4'), ('kind', '<i4', (4,)), ('index', '<i4', (4,)), ('pad', '<i4')])
KRAUS_DTYPE = np.dtype([('k', '<f8', (4, 8)), ('n_ops', '<i4'), ('qubit', '<i4')])


def lib():
    """Load libqcmrf_b200.so (built in-tree by qcmrf_b200.build / __graft_entry__.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError('qcmrf_b200: CUDA engine %s is not built (run `python -m qcmrf_b200.build`); '
                           'there is no CPU fallback' % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    vp, i32, u64, dbl = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint64, ctypes.c_double
    L.qcm_abi_version.restype = i32
    L.qcm_device_count.argtypes = [ctypes.POINTER(i32)]
    L.qcm_last_error.argtypes = [vp]
    L.qcm_last_error.restype = ctypes.c_char_p
    L.qcm_create.argtypes = [ctypes.POINTER(vp), i32, i32, i32, vp, vp]
    L.qcm_destroy.argtypes = [vp]
    L.qcm_set_shard.argtypes = [vp, i32, u64]
    L.qcm_get_amplitudes.argtypes = [vp, u64, u64, vp]
    L.qcm_set_amplitudes.argtypes = [vp, u64, u64, vp, i32]
    L.qcm_synchronize.argtypes = [vp]
    L.qcm_run_program.argtypes = [vp, vp, i32, vp, ctypes.c_size_t]
    L.qcm_postselect.argtypes = [vp, u64, u64, i32, vp, ctypes.POINTER(dbl)]
    L.qcm_sample.argtypes = [vp, u64, u64, u64, vp, i32, vp]
    L.qcm_sample_prepare.argtypes = [vp, ctypes.POINTER(dbl)]
    L.qcm_sample_sharded.argtypes = [vp, u64, u64, u64, vp, i32, vp, i32, vp, vp]
    L.qcm_small_max_qubits.argtypes = [i32]
    L.qcm_run_batch_small.argtypes = [i32, i32, i32, vp, vp, vp, vp, ctypes.c_size_t, vp, vp, vp, vp, vp, vp,
                                      u64, u64, vp, vp, vp, ctypes.POINTER(dbl)]
    L.qcm_run_batch_small_readout.argtypes = [i32, i32, i32, vp, vp, vp, vp, ctypes.c_size_t, vp, vp, vp, vp, vp, vp, vp,
                                              u64, u64, vp, vp, vp, ctypes.POINTER(dbl)]
    L.qcm_run_noisy_small.argtypes = [i32, i32, i32, vp, vp, vp, vp, i32, vp, vp, vp, vp, u64, u64, vp, ctypes.POINTER(dbl)]
    L.qcm_run_noisy_small_kraus.argtypes = [i32, i32, i32, vp, vp, vp, vp, i32, vp, i32, vp, i32, vp, vp, vp, vp, u64,
                                            u64, vp, ctypes.POINTER(dbl)]
    L.qcm_state_ptr.argtypes = [vp, ctypes.POINTER(vp), ctypes.POINTER(u64)]
    L.qcm_tree_level.argtypes = [vp, i32, ctypes.POINTER(vp), ctypes.POINTER(u64), ctypes.POINTER(i32)]
    L.qcm_set_active.argtypes = [vp, i32]
    L.qcm_get_active.argtypes = [vp, ctypes.POINTER(i32)]
    L.qcm_get_timing.argtypes = [vp, ctypes.POINTER(QcmTiming)]
    L.qcm_get_op_profile.argtypes = [vp, i32, vp, vp, vp, vp, ctypes.POINTER(i32)]
    L.qcm_postselect_device.argtypes = [vp, u64, u64, i32, vp, vp]
    L.qcm_sample_sharded_device.argtypes = [vp, u64, u64, u64, vp, i32, vp, i32, vp, vp]
    L.qcm_run_gather_block.argtypes = [vp, vp, i32, vp, ctypes.c_size_t, vp, i32, vp]
    L.qcm_enable_peer_access.argtypes = [i32, i32]
    L.qcm_ipc_export.argtypes = [i32, vp, vp, vp]
    L.qcm_ipc_open.argtypes = [i32, vp, vp]
    L.qcm_ipc_close.argtypes = [i32, vp]
    L.qcm_op_kernel_name.argtypes = [vp, i32]
    L.qcm_sample_released.argtypes = [vp, u64, u64, u64, i32, vp, vp, i32, vp, vp, ctypes.c_int64, vp, vp, i32, vp]
    L.qcm_op_kernel_name.restype = ctypes.c_char_p
    L.qcm_create_batched.argtypes = [ctypes.POINTER(vp), i32, i32, i32, i32, vp, vp]
    L.qcm_batch_size.argtypes = [vp, ctypes.POINTER(i32)]
    L.qcm_batch_select.argtypes = [vp, i32]
    L.qcm_postselect_resident.argtypes = [vp, u64, u64, i32, vp]
    L.qcm_fetch_probs.argtypes = [vp, i32, u64, u64, vp]
    L.qcm_sample_batched.argtypes = [vp, u64, u64, vp, vp, i32, vp]
    L.qcm_set_deferred.argtypes = [vp, i32]
    L.qcm_mark.argtypes = [vp, ctypes.POINTER(u64)]
    L.qcm_wait.argtypes = [vp, u64]
    L.qcm_tree_total_device.argtypes = [vp, vp]
    L.qcm_host_alloc.argtypes = [ctypes.POINTER(vp), ctypes.c_size_t]
    L.qcm_host_free.argtypes = [vp]
    L.qcm_gather_flag_words.argtypes = [i32, i32, i32, ctypes.POINTER(u64)]
    L.qcm_run_gather_block_inplace.argtypes = [vp, vp, i32, vp, ctypes.c_size_t, vp, i32, vp, u64, ctypes.c_uint32]
    L.qcm_mrf_exact.argtypes = [i32, i32, i32, vp, vp, vp, ctypes.POINTER(dbl), vp, vp, ctypes.POINTER(dbl)]
    L.qcm_mrf_last_error.restype = ctypes.c_char_p
    L.qcm_sample_sharded_devmass.argtypes = [vp, u64, u64, u64, vp, ctypes.c_int64, i32, vp, i32, vp, vp]
    L.qcm_sample_released_batched.argtypes = [vp, u64, u64, vp, i32, vp, vp, i32, vp, vp, ctypes.c_int64, vp, vp, i32, vp]
    if L.qcm_abi_version() != 1:
        raise RuntimeError('qcmrf_b200: ABI version mismatch')
    assert OP_DTYPE.itemsize == 72, OP_DTYPE.itemsize
    assert GATE_DTYPE.itemsize == 80 and CHANNEL_DTYPE.itemsize == 144
    _lib = L
    return L


def enable_peer_access(device, peer):
    """Let kernels running on `device` dereference pointers into `peer`'s memory (NVLink P2P)."""
    rc = lib().qcm_enable_peer_access(int(device), int(peer))
    if rc:
        raise NativeError(rc, (lib().qcm_last_error(None) or b'').decode())


def _check_global(rc):
    if rc:
        raise NativeError(rc, (lib().qcm_last_error(None) or b'').decode())


def ipc_export(device, dev_ptr):
    """(handle bytes, offset) of the cudaMalloc allocation containing dev_ptr (qcm_ipc_export)."""
    hd = (ctypes.c_ubyte * 64)()
    off = ctypes.c_uint64()
    _check_global(lib().qcm_ipc_export(int(device), ctypes.c_void_p(int(dev_ptr)), hd, ctypes.byref(off)))
    return bytes(hd), off.value


def ipc_open(device, handle):
    """Map an exported allocation for kernels on `device`; returns its base address in this process."""
    hd = (ctypes.c_ubyte * 64).from_buffer_copy(handle)
    base = ctypes.c_void_p()
    _check_global(lib().qcm_ipc_open(int(device), hd, ctypes.byref(base)))
    return base.value


def ipc_close(device, base):
    _check_global(lib().qcm_ipc_close(int(device), ctypes.c_void_p(int(base))))


def device_count():
    n = ctypes.c_int(0)
    rc = lib().qcm_device_count(ctypes.byref(n))
    return n.value if rc == 0 else 0


def _ptr(a):
    return None if a is None else a.ctypes.data


class Handle:
    """One statevector on one GPU (see qcm_create) -- or, with batch > 1, the `batch` states of a sweep in one
    allocation, every kernel of a program launched once for all of them (qcm_create_batched)."""

    def __init__(self, n_local, precision='single', device=0, ext_state_ptr=None, ext_stream=None, batch=1):
        self._h = ctypes.c_void_p()
        self.batch = int(batch)
        self.generation = 0                      # bumped by every post-selection: lazily fetched pmfs check it
        self.deferred = False                    # set_deferred: calls only enqueue
        self.n_local = int(n_local)
        self.prec = QCM_C64 if precision in ('single', 'c64', 32) else QCM_C128
        self.cdtype = np.complex64 if self.prec == QCM_C64 else np.complex128
        L = lib()
        rc = L.qcm_create_batched(ctypes.byref(self._h), int(device), self.n_local, self.prec, self.batch,
                                  ctypes.c_void_p(ext_state_ptr), ctypes.c_void_p(ext_stream))
        if rc:
            self._h = ctypes.c_void_p()
            raise NativeError(rc, (L.qcm_last_error(None) or b'').decode())

    def _check(self, rc):
        if rc:
            raise NativeError(rc, (lib().qcm_last_error(self._h) or b'').decode())

    def close(self):
        if self._h:
            lib().qcm_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_shard(self, n_global, rank):
        self._check(lib().qcm_set_shard(self._h, int(n_global), int(rank)))

    def run_program(self, ops, tables):
        """tables: the program's coefficient tables; a batched handle takes shape (batch, n_tables), one row per point."""
        ops = np.ascontiguousarray(ops, dtype=OP_DTYPE)
        tables = np.ascontiguousarray(tables, dtype=np.float64)
        if self.batch > 1 and (tables.ndim != 2 or tables.shape[0] != self.batch):
            raise ValueError('batched handle: tables must have shape (batch, n_tables)')
        self._check(lib().qcm_run_program(self._h, _ptr(ops), len(ops), _ptr(tables), tables.size // self.batch))

    def postselect(self, mask, value, n_out_bits, want_probs=True, out=None):
        """(probs, kept); a batched handle returns arrays of shape (batch, 2^n_out_bits) and (batch,).
        out = (probs, kept) page-locked arrays (deferred mode: valid after synchronize() / wait()); returns them."""
        self.generation += 1
        if out is not None:
            probs, kept = out
            self._check(lib().qcm_postselect(self._h, int(mask), int(value), int(n_out_bits), _ptr(probs) if want_probs else None,
                                             kept.ctypes.data_as(ctypes.POINTER(ctypes.c_double))))
            return probs, kept
        if self.batch > 1:
            probs = np.empty((self.batch, 1 << n_out_bits), dtype=np.float64) if want_probs else None
            kept = np.empty(self.batch, dtype=np.float64)
            self._check(lib().qcm_postselect(self._h, int(mask), int(value), int(n_out_bits), _ptr(probs),
                                             kept.ctypes.data_as(ctypes.POINTER(ctypes.c_double))))
            return probs, kept
        probs = np.empty(1 << n_out_bits, dtype=np.float64) if want_probs else None
        kept = ctypes.c_double()
        self._check(lib().qcm_postselect(self._h, int(mask), int(value), int(n_out_bits), _ptr(probs),
                                         ctypes.byref(kept)))
        return probs, kept.value

    def postselect_resident(self, mask, value, n_out_bits, out=None):
        """kept (array of `batch`); the probability blocks stay on the device until the next post-selection on this
        handle (fetch_probs copies one out)."""
        self.generation += 1
        kept = np.empty(self.batch, dtype=np.float64) if out is None else out
        self._check(lib().qcm_postselect_resident(self._h, int(mask), int(value), int(n_out_bits), _ptr(kept)))
        return kept

    def fetch_probs(self, point, n_out_bits, first=0, count=None):
        if count is None:
            count = (1 << n_out_bits) - first
        out = np.empty(int(count), dtype=np.float64)
        self._check(lib().qcm_fetch_probs(self._h, int(point), int(first), int(count), _ptr(out)))
        return out

    def tree_total_device(self, dev_ptr):
        """qcm_tree_total_device: the local state's total |amp|^2 written to a device double, in stream order."""
        self._check(lib().qcm_tree_total_device(self._h, ctypes.c_void_p(dev_ptr)))

    def set_deferred(self, flag):
        """Deferred mode: calls enqueue and return; pass page-locked output arrays (pinned_empty) and call synchronize()."""
        self._check(lib().qcm_set_deferred(self._h, 1 if flag else 0))
        self.deferred = bool(flag)

    def batch_select(self, point):
        self._check(lib().qcm_batch_select(self._h, int(point)))

    def sample_batched(self, shots, seed, stream_ids, clbit_qubit=None, out=None):
        keys = np.empty((self.batch, int(shots)), dtype=np.uint64) if out is None else out
        sid = np.ascontiguousarray(stream_ids, dtype=np.uint64)
        assert sid.size == self.batch
        cq = None if clbit_qubit is None else np.ascontiguousarray(clbit_qubit, dtype=np.int32)
        self._check(lib().qcm_sample_batched(self._h, int(shots), int(seed), _ptr(sid), _ptr(cq),
                                             0 if cq is None else len(cq), _ptr(keys)))
        return keys

    def sample_released_batched(self, shots, seed, stream_ids, n_ctrl, ctrl, p1, p1_off, vclbit, clbit_pos, n_clbits, out=None):
        """p1: (batch, n_p1) released-qubit probability tables, one row per sweep point."""
        keys = np.empty((self.batch, int(shots)), dtype=np.uint64) if out is None else out
        sid = np.ascontiguousarray(stream_ids, dtype=np.uint64)
        p1 = np.ascontiguousarray(p1, dtype=np.float64)
        assert sid.size == self.batch and p1.shape[0] == self.batch
        self._check(lib().qcm_sample_released_batched(self._h, int(shots), int(seed), _ptr(sid), len(n_ctrl), _ptr(n_ctrl),
                                                      _ptr(ctrl), int(ctrl.shape[1]), _ptr(p1), _ptr(p1_off), int(p1.shape[1]),
                                                      _ptr(vclbit), _ptr(clbit_pos), int(n_clbits), _ptr(keys)))
        return keys

    def mark(self):
        """qcm_mark: ticket of a point in the handle's stream behind everything enqueued so far."""
        t = ctypes.c_uint64()
        self._check(lib().qcm_mark(self._h, ctypes.byref(t)))
        return t.value

    def wait(self, ticket):
        """qcm_wait: block until the marked point has been reached (later work keeps running)."""
        self._check(lib().qcm_wait(self._h, int(ticket)))

    def sample(self, shots, seed, stream_id=0, clbit_qubit=None, out=None):
        keys = np.empty(int(shots), dtype=np.uint64) if out is None else out
        cq = None if clbit_qubit is None else np.ascontiguousarray(clbit_qubit, dtype=np.int32)
        self._check(lib().qcm_sample(self._h, int(shots), int(seed), int(stream_id), _ptr(cq),
                                     0 if cq is None else len(cq), _ptr(keys)))
        return keys

    def sample_released(self, shots, seed, stream_id, n_ctrl, ctrl, p1, p1_off, vclbit, clbit_pos, n_clbits):
        """qcm_sample_released: full-width keys of a release-width circuit, released qubits drawn on the device."""
        keys = np.empty(int(shots), dtype=np.uint64)
        self._check(lib().qcm_sample_released(self._h, int(shots), int(seed), int(stream_id), len(n_ctrl), _ptr(n_ctrl),
                                              _ptr(ctrl), int(ctrl.shape[1]), _ptr(p1), _ptr(p1_off), int(p1.size),
                                              _ptr(vclbit), _ptr(clbit_pos), int(n_clbits), _ptr(keys)))
        return keys

    def run_gather_block(self, ops, tables, src_slab_ptrs, dst_ptr):
        """qcm_run_gather_block: fused qubit swap + blocked pass reading the peers' shards."""
        ops = np.ascontiguousarray(ops, dtype=OP_DTYPE)
        tables = np.ascontiguousarray(tables, dtype=np.float64)
        src = (ctypes.c_void_p * len(src_slab_ptrs))(*[ctypes.c_void_p(int(p)) for p in src_slab_ptrs])
        s = len(src_slab_ptrs).bit_length() - 1
        self._check(lib().qcm_run_gather_block(self._h, _ptr(ops), len(ops), _ptr(tables), tables.size, src, s,
                                               ctypes.c_void_p(int(dst_ptr))))

    def run_gather_block_inplace(self, ops, tables, src_slab_ptrs, flag_ptrs, flag_words, epoch):
        """qcm_run_gather_block_inplace: the fused qubit swap + blocked pass writing over this rank's own slabs."""
        ops = np.ascontiguousarray(ops, dtype=OP_DTYPE)
        tables = np.ascontiguousarray(tables, dtype=np.float64)
        src = (ctypes.c_void_p * len(src_slab_ptrs))(*[ctypes.c_void_p(int(p)) for p in src_slab_ptrs])
        fl = (ctypes.c_void_p * len(flag_ptrs))(*[ctypes.c_void_p(int(p)) for p in flag_ptrs])
        s = len(src_slab_ptrs).bit_length() - 1
        self._check(lib().qcm_run_gather_block_inplace(self._h, _ptr(ops), len(ops), _ptr(tables), tables.size, src, s, fl,
                                                       int(flag_words), int(epoch)))

    def postselect_device(self, mask, value, n_out_bits, dev_probs_ptr, dev_kept_ptr):
        """qcm_postselect_device: results stay on the GPU (device pointers), no synchronisation."""
        self._check(lib().qcm_postselect_device(self._h, int(mask), int(value), int(n_out_bits),
                                                ctypes.c_void_p(dev_probs_ptr), ctypes.c_void_p(dev_kept_ptr)))

    def sample_sharded_device(self, shots, seed, stream_id, rank_masses, clbit_qubit, dev_keys_ptr, dev_mine_ptr):
        rm = np.ascontiguousarray(rank_masses, dtype=np.float64)
        cq = None if clbit_qubit is None else np.ascontiguousarray(clbit_qubit, dtype=np.int32)
        self._check(lib().qcm_sample_sharded_device(self._h, int(shots), int(seed), int(stream_id), _ptr(rm), len(rm),
                                                    _ptr(cq), 0 if cq is None else len(cq),
                                                    ctypes.c_void_p(dev_keys_ptr), ctypes.c_void_p(dev_mine_ptr)))

    def sample_sharded_devmass(self, shots, seed, stream_id, dev_masses_ptr, mass_stride, n_ranks, clbit_qubit, dev_keys_ptr,
                               dev_mine_ptr):
        """qcm_sample_sharded_devmass: rank masses read on the device (no host round trip after the all-gather)."""
        cq = None if clbit_qubit is None else np.ascontiguousarray(clbit_qubit, dtype=np.int32)
        self._check(lib().qcm_sample_sharded_devmass(self._h, int(shots), int(seed), int(stream_id), ctypes.c_void_p(dev_masses_ptr),
                                                     int(mass_stride), int(n_ranks), _ptr(cq), 0 if cq is None else len(cq),
                                                     ctypes.c_void_p(dev_keys_ptr), ctypes.c_void_p(dev_mine_ptr)))

    def sample_prepare(self):
        m = ctypes.c_double()
        self._check(lib().qcm_sample_prepare(self._h, ctypes.byref(m)))
        return m.value

    def sample_sharded(self, shots, seed, stream_id, rank_masses, clbit_qubit=None):
        keys = np.empty(int(shots), dtype=np.uint64)
        mine = np.empty(int(shots), dtype=np.uint8)
        rm = np.ascontiguousarray(rank_masses, dtype=np.float64)
        cq = None if clbit_qubit is None else np.ascontiguousarray(clbit_qubit, dtype=np.int32)
        self._check(lib().qcm_sample_sharded(self._h, int(shots), int(seed), int(stream_id), _ptr(rm), len(rm),
                                             _ptr(cq), 0 if cq is None else len(cq), _ptr(keys), _ptr(mine)))
        return keys, mine.astype(bool)

    def get_amplitudes(self, first=0, count=None):
        if count is None:
            count = (1 << self.n_local) - first
        out = np.empty(int(count), dtype=self.cdtype)
        self._check(lib().qcm_get_amplitudes(self._h, int(first), int(count), _ptr(out)))
        return out

    def set_amplitudes(self, amps, first=0, n_active=None):
        amps = np.ascontiguousarray(amps, dtype=self.cdtype)
        self._check(lib().qcm_set_amplitudes(self._h, int(first), amps.size, _ptr(amps),
                                             self.n_local if n_active is None else int(n_active)))

    def set_active(self, n_active):
        self._check(lib().qcm_set_active(self._h, int(n_active)))

    def get_active(self):
        v = ctypes.c_int()
        self._check(lib().qcm_get_active(self._h, ctypes.byref(v)))
        return v.value

    def state_ptr(self):
        p, b = ctypes.c_void_p(), ctypes.c_uint64()
        self._check(lib().qcm_state_ptr(self._h, ctypes.byref(p), ctypes.byref(b)))
        return p.value, b.value

    def tree_level(self, level):
        """(device pointer, entry count, number of levels) of one level of the sampler's sum tree, read-only: 0 = the
        chunk sums ... top, -1 = the finer level under level 0.  Builds nothing; raises when there is no such level."""
        p, n, nl = ctypes.c_void_p(), ctypes.c_uint64(), ctypes.c_int()
        self._check(lib().qcm_tree_level(self._h, int(level), ctypes.byref(p), ctypes.byref(n), ctypes.byref(nl)))
        return p.value, n.value, nl.value

    def synchronize(self):
        self._check(lib().qcm_synchronize(self._h))

    def op_profile(self):
        """[(kind, ms, bytes_read, bytes_written)] for every launch of the last program."""
        n = ctypes.c_int()
        self._check(lib().qcm_get_op_profile(self._h, 0, None, None, None, None, ctypes.byref(n)))
        k = np.zeros(n.value, dtype=np.int32); ms = np.zeros(n.value, dtype=np.float32)
        rd = np.zeros(n.value, dtype=np.uint64); wr = np.zeros(n.value, dtype=np.uint64)
        self._check(lib().qcm_get_op_profile(self._h, n.value, _ptr(k), _ptr(ms), _ptr(rd), _ptr(wr), ctypes.byref(n)))
        return [(int(a), float(b), int(c), int(d)) for a, b, c, d in zip(k, ms, rd, wr)]

    def op_kernels(self):
        """Kernel name per op of the last program (same indices as op_profile; '' where not recorded)."""
        n = ctypes.c_int()
        self._check(lib().qcm_get_op_profile(self._h, 0, None, None, None, None, ctypes.byref(n)))
        return [(lib().qcm_op_kernel_name(self._h, i) or b'').decode() for i in range(n.value)]

    def timing(self):
        t = QcmTiming()
        self._check(lib().qcm_get_timing(self._h, ctypes.byref(t)))
        return {f: getattr(t, f) for f, _ in QcmTiming._fields_}


def small_max_qubits(precision='double'):
    return lib().qcm_small_max_qubits(QCM_C64 if precision in ('single', 'c64', 32) else QCM_C128)


def run_batch_small(plans, clbit_maps, ps, shots, seed, precision='double', device=0, want_probs=True,
                    stream_ids=None, readout=None):
    """plans: list of fusion.Plan (fully materialised); clbit_maps: list of int arrays
    (clbit -> physical qubit or -1); ps: list of (mask, value, bits); readout: None or (n, 64, 2) per-clbit flip
    probabilities applied to the keys on the device (qcm_run_batch_small_readout).  Returns
    (keys[n][shots] uint64, probs list, kept array, device_ms)."""
    n = len(plans)
    nq = np.array([p.n_phys for p in plans], dtype=np.int32)
    op_begin = np.zeros(n + 1, dtype=np.int64)
    ops, tabs, toff = [], [], 0
    for i, p in enumerate(plans):
        o = p.ops.copy()
        o['table_off'] += toff
        ops.append(o)
        tabs.append(p.tables)
        toff += p.tables.size
        op_begin[i + 1] = op_begin[i] + len(o)
    ops = np.concatenate(ops) if ops else np.zeros(0, dtype=OP_DTYPE)
    tabs = np.concatenate(tabs) if tabs else np.zeros(0)
    cq = np.full((n, 64), -1, dtype=np.int32)
    ncl = np.zeros(n, dtype=np.int32)
    for i, m in enumerate(clbit_maps):
        cq[i, :len(m)] = m
        ncl[i] = len(m)
    pm = np.array([int(x[0]) for x in ps], dtype=np.uint64)
    pv = np.array([int(x[1]) for x in ps], dtype=np.uint64)
    pb = np.array([int(x[2]) for x in ps], dtype=np.int32)
    keys = np.empty((n, int(shots)), dtype=np.uint64) if shots else None
    pbeg = np.concatenate([[0], np.cumsum(1 << pb.astype(np.int64))])
    probs = np.empty(int(pbeg[-1]), dtype=np.float64) if want_probs else None
    kept = np.empty(n, dtype=np.float64)
    ms = ctypes.c_double()
    prec = QCM_C64 if precision in ('single', 'c64', 32) else QCM_C128
    sid = None if stream_ids is None else np.ascontiguousarray(stream_ids, dtype=np.uint64)
    if readout is None:
        rc = lib().qcm_run_batch_small(int(device), prec, n, _ptr(nq), _ptr(op_begin), _ptr(ops), _ptr(tabs), tabs.size,
                                       _ptr(cq), _ptr(ncl), _ptr(pm), _ptr(pv), _ptr(pb), _ptr(sid), int(shots), int(seed),
                                       _ptr(keys), _ptr(probs), _ptr(kept), ctypes.byref(ms))
    else:
        ro = np.ascontiguousarray(readout, dtype=np.float64)
        assert ro.shape == (n, 64, 2), ro.shape
        rc = lib().qcm_run_batch_small_readout(int(device), prec, n, _ptr(nq), _ptr(op_begin), _ptr(ops), _ptr(tabs),
                                               tabs.size, _ptr(cq), _ptr(ncl), _ptr(ro), _ptr(pm), _ptr(pv), _ptr(pb),
                                               _ptr(sid), int(shots), int(seed), _ptr(keys), _ptr(probs), _ptr(kept),
                                               ctypes.byref(ms))
    if rc:
        raise NativeError(rc, 'qcm_run_batch_small failed')
    plist = [probs[pbeg[i]:pbeg[i + 1]] for i in range(n)] if want_probs else None
    return keys, plist, kept, ms.value


def _noisy_records(encoded, kraus):
    """Flat qcm_gate, qcm_channel (and for `kraus`, qcm_gate_error and qcm_kraus) arrays of noise.EncodedNoise
    programs, record indices made global; with the per-circuit clbit maps and readout tables."""
    n = len(encoded)
    nq = np.array([e.n_qubits for e in encoded], dtype=np.int32)
    gate_begin = np.concatenate([[0], np.cumsum([e.n_gates for e in encoded])]).astype(np.int64)
    gates = np.zeros(int(gate_begin[-1]), dtype=GATE_DTYPE)
    chans, errs, krs = [], [], []
    coff = eoff = koff = 0
    for i, e in enumerate(encoded):
        g = gates[gate_begin[i]:gate_begin[i + 1]]
        g['m'], g['target'], g['ctrl_mask'], g['ctrl_value'] = e.matrix, e.target, e.ctrl_mask, e.ctrl_value
        g['channel'] = np.where(e.channel >= 0, e.channel + (eoff if kraus else coff), -1)
        ch = np.zeros(len(e.n_paulis), dtype=CHANNEL_DTYPE)
        ch['cum'], ch['n_paulis'], ch['qubit'] = e.cum, e.n_paulis, e.chan_qubits
        chans.append(ch)
        if kraus:
            er = np.zeros(len(e.err_n_stages), dtype=GATE_ERROR_DTYPE)
            er['n_stages'], er['kind'] = e.err_n_stages, e.err_kind
            er['index'] = e.err_index + np.where(e.err_kind == 1, koff, coff)
            kr = np.zeros(len(e.kraus_n_ops), dtype=KRAUS_DTYPE)
            kr['k'], kr['n_ops'], kr['qubit'] = e.kraus_ops, e.kraus_n_ops, e.kraus_qubit
            errs.append(er)
            krs.append(kr)
            eoff += len(er)
            koff += len(kr)
        coff += len(ch)
    cat = lambda parts, dt: np.concatenate(parts) if parts else np.zeros(0, dtype=dt)
    cq = np.full((n, 64), -1, dtype=np.int32)
    ncl = np.zeros(n, dtype=np.int32)
    ro = np.zeros((n, 64, 2))
    for i, e in enumerate(encoded):
        cq[i, :e.n_clbits] = e.clbit_map
        ncl[i] = e.n_clbits
        ro[i] = e.readout
    return (nq, gate_begin, gates, cat(chans, CHANNEL_DTYPE), cat(errs, GATE_ERROR_DTYPE), cat(krs, KRAUS_DTYPE),
            cq, ncl, ro)


def run_noisy_small(encoded, shots, seed, precision='double', device=0, stream_ids=None):
    """Noisy shots of noise.EncodedNoise programs whose errors are single Pauli channels (qcm_run_noisy_small): one
    trajectory per shot.  Returns (keys[n][shots] uint64, device_ms)."""
    nq, gate_begin, gates, channels, _, _, cq, ncl, ro = _noisy_records(encoded, False)
    keys = np.empty((len(encoded), int(shots)), dtype=np.uint64)
    sid = None if stream_ids is None else np.ascontiguousarray(stream_ids, dtype=np.uint64)
    ms = ctypes.c_double()
    prec = QCM_C64 if precision in ('single', 'c64', 32) else QCM_C128
    rc = lib().qcm_run_noisy_small(int(device), prec, len(encoded), _ptr(nq), _ptr(gate_begin), _ptr(gates),
                                   _ptr(channels), len(channels), _ptr(cq), _ptr(ncl), _ptr(ro) if ro.any() else None,
                                   _ptr(sid), int(shots), int(seed), _ptr(keys), ctypes.byref(ms))
    if rc:
        raise NativeError(rc, 'qcm_run_noisy_small failed')
    return keys, ms.value


def run_noisy_small_kraus(encoded, shots, seed, precision='double', device=0, stream_ids=None):
    """Noisy shots of noise.EncodedNoise programs through their error records (qcm_run_noisy_small_kraus): errors
    of up to 4 stages, Pauli or 1-qubit Kraus.  Any encoding runs here (a Pauli-only one as one-stage records).
    Returns (keys[n][shots] uint64, device_ms)."""
    nq, gate_begin, gates, channels, errors, krauses, cq, ncl, ro = _noisy_records(encoded, True)
    keys = np.empty((len(encoded), int(shots)), dtype=np.uint64)
    sid = None if stream_ids is None else np.ascontiguousarray(stream_ids, dtype=np.uint64)
    ms = ctypes.c_double()
    prec = QCM_C64 if precision in ('single', 'c64', 32) else QCM_C128
    rc = lib().qcm_run_noisy_small_kraus(int(device), prec, len(encoded), _ptr(nq), _ptr(gate_begin), _ptr(gates),
                                         _ptr(errors), len(errors),
                                         _ptr(channels), len(channels), _ptr(krauses), len(krauses), _ptr(cq),
                                         _ptr(ncl), _ptr(ro) if ro.any() else None, _ptr(sid), int(shots), int(seed),
                                         _ptr(keys), ctypes.byref(ms))
    if rc:
        raise NativeError(rc, 'qcm_run_noisy_small_kraus failed')
    return keys, ms.value


def mrf_exact(cliques, weights, n=None, want_pmf=True, want_energies=False, device=0):
    """qcm_mrf_exact: (ln Z, pmf or None, energies or None, device ms) of a binary MRF by enumeration on the GPU;
    state id with x_0 as its most significant bit, weights clique-major in itertools.product order."""
    if n is None:
        n = max(max(c) for c in cliques) + 1
    size = np.array([len(c) for c in cliques], dtype=np.int32)
    var = np.array([v for c in cliques for v in c], dtype=np.int32)
    w = np.ascontiguousarray(weights, dtype=np.float64)
    if w.size != int(sum(1 << int(m) for m in size)):
        raise ValueError('weights: %d entries, the cliques need %d' % (w.size, sum(1 << int(m) for m in size)))
    pmf = np.empty(1 << n, dtype=np.float64) if want_pmf else None
    en = np.empty(1 << n, dtype=np.float64) if want_energies else None
    lz, ms = ctypes.c_double(), ctypes.c_double()
    rc = lib().qcm_mrf_exact(int(device), int(n), len(size), _ptr(size), _ptr(var), _ptr(w), ctypes.byref(lz), _ptr(pmf), _ptr(en),
                             ctypes.byref(ms))
    if rc:
        raise NativeError(rc, (lib().qcm_mrf_last_error() or b'').decode())
    return lz.value, pmf, en, ms.value


def gather_flag_words(n_local, s, precision):
    """Entries (uint32) of one rank's flag array for qcm_run_gather_block_inplace."""
    w = ctypes.c_uint64()
    _check_global(lib().qcm_gather_flag_words(int(n_local), int(s), QCM_C64 if precision in ('single', 'c64', 32) else QCM_C128,
                                              ctypes.byref(w)))
    return w.value


class PinnedArray:
    """A numpy array over page-locked host memory (qcm_host_alloc): the target of asynchronous device->host copies.
    The memory is freed when this object is collected; `array` must not outlive it."""

    def __init__(self, shape, dtype):
        dtype = np.dtype(dtype)
        n = int(np.prod(shape)) * dtype.itemsize
        p = ctypes.c_void_p()
        _check_global(lib().qcm_host_alloc(ctypes.byref(p), n))
        self._p = p
        buf = (ctypes.c_ubyte * max(n, 1)).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def __del__(self):
        try:
            if self._p:
                lib().qcm_host_free(self._p)
                self._p = None
        except Exception:
            pass
