"""Every kernel path of the large-state engine against the numpy statement of the op semantics
(tests/engine_emulator.run_plan, complex128).

The engine picks its kernel at run time (plan_block / launch_block_plan / try_lowq in qcm_api.cu), and several
kernels choose again inside: 32-bit index arithmetic when every index qubit is below 32, and grid-stride loops that
only iterate when the grid is capped.  The corpus below is built so that every launcher instantiation runs
(the kernel census), and it runs on plain handles, with index qubits far above 32 (a sharded handle's global
qubits), on batched handles with per-point tables, and in child processes under each launch knob.  States past
2^31 and 2^32 amplitudes are checked against a factorised reference: every op touches a small qubit set T of a
product state, so the state is (product over the other qubits) x (a 2^|T| state) exactly.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
if __name__ == '__main__':                                   # child process of the knob matrix
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.dirname(HERE))

import engine_emulator as em                                # noqa: E402
from qcmrf_b200 import _native, fusion                      # noqa: E402

F = fusion
TOL_AMP = {'double': 1e-12, 'single': 3e-6}
TOL_REL = {'double': 1e-9, 'single': 2e-4}


def _has_cuda():
    try:
        return _native.device_count() > 0
    except Exception:
        return False


pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not _has_cuda(), reason='needs a CUDA device')]


def weissman_tv_bound(K, S, alpha=1e-6):
    """P(TV > bound) <= alpha for S draws over K outcomes."""
    return 0.5 * np.sqrt(2.0 * (K * np.log(2.0) + np.log(1.0 / alpha)) / S)


class _P:
    pass


def _plan(ops, tabs, n):
    pl = _P()
    pl.ops, pl.tables, pl.n_phys = ops, tabs, n
    return pl


# ---- program builder ---------------------------------------------------------------------------------------
class Prog:
    """Engine program over n_local stored qubits, tracking the materialised count; tables are random (unitary
    multiplexer tables, unit-modulus diagonals) so that every program preserves the norm."""

    def __init__(self, rng, n_local):
        self.e = F._Emitter()
        self.rng = rng
        self.n = n_local
        self.act = 0
        self.flag_last = False

    def u(self, m):
        q, _ = np.linalg.qr(self.rng.randn(1 << m, 2, 2) + 1j * self.rng.randn(1 << m, 2, 2))
        return q

    def d(self, m):
        return np.exp(1j * self.rng.uniform(0, 2 * np.pi, 1 << m))

    def init(self, n0, qv=None):
        if qv is None:
            v = self.rng.randn(max(n0, 1), 2) + 1j * self.rng.randn(max(n0, 1), 2)
            v /= np.linalg.norm(v, axis=1, keepdims=True)
            qv = np.stack([v[:, 0].real, v[:, 0].imag, v[:, 1].real, v[:, 1].imag], axis=1)
        self.e.op(F.QCM_OP_INIT_PRODUCT, n_in=0, n_out=n0, table_off=self.e.table(qv))
        self.act = n0
        return self

    def mux(self, t, ctrl):
        n_out = max(self.act, t + 1)
        self.e.op(F.QCM_OP_MUX1Q, target=t, ctrl=list(ctrl), n_in=self.act, n_out=n_out,
                  table_off=self.e.table(F._mux_table_f64(self.u(len(ctrl)))))
        self.act = n_out
        return self

    def block(self, tq, members):
        """members: ('m', target, ctrl) or ('d', ctrl); targets new qubits act.. are materialised."""
        tq = sorted(tq)
        n_out = max(self.act, tq[-1] + 1)
        self.e.op(F.QCM_OP_BLOCK, target=len(tq), ctrl=tq, n_in=self.act, n_out=n_out, n_ctrl=len(members))
        for mb in members:
            if mb[0] == 'm':
                self.e.op(F.QCM_OP_MUX1Q, target=mb[1], ctrl=list(mb[2]), n_in=self.act, n_out=n_out,
                          table_off=self.e.table(F._mux_table_f64(self.u(len(mb[2])))))
            else:
                self.e.op(F.QCM_OP_DIAG, ctrl=list(mb[1]), n_in=self.act, n_out=n_out,
                          table_off=self.e.table(F._diag_table_f64(self.d(len(mb[1])))))
        self.act = n_out
        return self

    def expand(self, M, ctrls, n_diag=0, diag_ctrl=()):
        """Materialise qubits act .. act+M-1, one MUX1Q each (ctrls[j] its index qubits), plus diagonal members."""
        tq = list(range(self.act, self.act + M))
        mem = [('m', t, c) for t, c in zip(tq, ctrls)] + [('d', list(diag_ctrl))] * n_diag
        if len(mem) == 1:
            return self.mux(tq[0], ctrls[0])
        return self.block(tq, mem)

    def diag(self, ctrl):
        self.e.op(F.QCM_OP_DIAG, ctrl=list(ctrl), n_in=self.act, n_out=self.act,
                  table_off=self.e.table(F._diag_table_f64(self.d(len(ctrl)))))
        return self

    def diag_block(self, ctrls):
        self.e.op(F.QCM_OP_BLOCK, target=0, ctrl=(), n_in=self.act, n_out=self.act, n_ctrl=len(ctrls))
        for c in ctrls:
            self.diag(c)
        return self

    def swap(self, a, b):
        self.e.op(F.QCM_OP_SWAP, target=a, ctrl=[b], n_in=self.act, n_out=self.act)
        return self

    def extend(self, n_out):
        self.e.op(F.QCM_OP_EXTEND, n_in=self.act, n_out=n_out)
        self.act = n_out
        return self

    def finish(self):
        ops, tabs = self.e.finish()
        if self.flag_last:
            F._flag_last_pass(ops)
        return ops, tabs


def _pick(rng, pool, k):
    pool = list(pool)
    return [int(x) for x in rng.permutation(pool)[:k]] if pool else []


# ---- the census corpus ------------------------------------------------------------------------------------
_U_BLOCK = {1: 4, 2: 2, 3: 1, 4: 1, 5: 1}
_U_EXPAND = {1: 4, 2: 4, 3: 2, 4: 2, 5: 2}


def census_names(precision):
    """Every kernel the launchers can record for an op of a program on an unsharded or sharded handle."""
    if precision == 'single':
        R = 'float'
        names = {'k_init<float,2>', 'k_init<float,1>', 'k_expand_tree<float,2>', 'k_expand_tree<float,1>',
                 'k_lowq<float,2,UB=3,MH=0>', 'k_lowq<float,2,UB=2,MH=1>', 'k_lowq<float,2,UB=1,MH=2>',
                 'k_diag<float,2,U=4>', 'k_diag<float,1,U=4>', 'k_diag_multi<float,2,U=4>', 'k_diag_multi<float,1,U=4>',
                 'k_diag<float,2,U=4> (diagonal block, one pass per member)', 'k_swap<float,2>', 'k_swap<float,1>',
                 'k_zero<float>'}
        names |= {'k_expand_low<float,2,MH=%d,TB=8,NW=8>' % mh for mh in range(3)}
        names |= {'k_expand<float,2,M=%d,U=%d,Q0=%d>' % (m, _U_EXPAND[m], q) for m in range(1, 6) for q in (0, 1)}
        names |= {'k_expand<float,1,M=%d,U=%d,Q0=0>' % (m, _U_EXPAND[m]) for m in range(1, 6)}
        Vs = (1, 2)
    else:
        R = 'double'
        names = {'k_init<double,1>', 'k_expand_tree<double,1>', 'k_lowq<double,1,UB=3,MH=0>', 'k_lowq<double,1,UB=2,MH=1>',
                 'k_lowq<double,1,UB=1,MH=2>', 'k_diag<double,1,U=4>', 'k_diag_multi<double,1,U=4>',
                 'k_diag<double,1,U=4> (diagonal block, one pass per member)', 'k_swap<double,1>', 'k_zero<double>'}
        names |= {'k_expand_low<double,1,MH=%d,TB=7,NW=4>' % mh for mh in range(4)}
        names |= {'k_expand<double,1,M=%d,U=%d,Q0=0>' % (m, _U_EXPAND[m]) for m in range(1, 6)}
        Vs = (1,)
    names |= {'k_block<%s,%d,M=%d,U=%d,LAZY=%d>' % (R, V, m, _U_BLOCK[m], lz) for V in Vs for m in range(1, 6) for lz in (0, 1)}
    return names


def census_corpus(precision, seed=0):
    """(n_local, ops, tables) programs that together reach every name of census_names(precision)."""
    rng = np.random.RandomState(seed)
    c64 = precision == 'single'
    out = []

    def add(p):
        ops, tabs = p.finish()
        out.append((p.n, ops, tabs))
    # expansions from 3 qubits: M = 1..4 through the precombined table, index qubits without and with qubit 0 (Q0)
    for q0 in (False, True):
        p = Prog(rng, 13).init(3)
        for M in (1, 2, 3, 4):
            base = [1, 2] if not q0 else [0, 2]
            p.expand(M, [base[:1 + (j % 2)] for j in range(M)])
        add(p)
    # M = 5 with five diagonal members: no product tree, the precombined table (Q0 both ways)
    for q0 in (False, True):
        p = Prog(rng, 9).init(4)
        p.expand(5, [[1, 3], [2], [], [3], [1]] if not q0 else [[0, 3], [2], [], [3], [1]], n_diag=5, diag_ctrl=[1, 2])
        add(p)
    # expansions out of a state of zero qubits (one amplitude: V = 1), M = 1..5 and a wide one (product tree)
    for M in (1, 2, 3, 4, 5, 6):
        p = Prog(rng, M + 1).init(0)
        p.expand(M, [[]] * M, n_diag=5 if M == 5 else 0, diag_ctrl=[])
        p.diag([0])
        add(p)
    # the product tree: M = 4 whose index-qubit union overflows the table (nu + M > 12), M = 5..8 in place of the table
    p = Prog(rng, 19).init(10)
    p.expand(4, [[0, 1, 2], [3, 4, 5], [6, 7], [8, 9]])
    p.expand(5, [_pick(rng, range(p.act), 2) for _ in range(5)], n_diag=2, diag_ctrl=[0, 5])
    add(p)
    # a wide last pass flagged for rotated output (k_expand_low), each loop depth
    for M in ((6, 7, 8) if c64 else (5, 6, 7, 8)):
        p = Prog(rng, 10 + M).init(10)
        p.expand(M, [_pick(rng, range(10), int(rng.randint(0, 3))) for _ in range(M)])
        p.flag_last = True
        add(p)
    # nu + M > 12 below M = 4: k_block materialises (LAZY); M = 1 / 2 also via a doubled target
    p = Prog(rng, 18).init(12)
    p.expand(3, [list(range(0, 10)), [10, 11], [1, 2]])
    p.block([p.act], [('m', p.act, [0, 1]), ('m', p.act, [2])])
    p.block([p.act, p.act + 1], [('m', p.act, [3]), ('m', p.act + 1, [0]), ('m', p.act, [5])])
    add(p)
    # a lazy block of one target at qubit 0 out of zero qubits (V = 1)
    p = Prog(rng, 4).init(0)
    p.block([0], [('m', 0, []), ('m', 0, [])])
    p.diag([0])
    add(p)
    # lazy blocks over an old target plus new ones, lowest target >= 1 (V = 2) and = 0 (V = 1), M = 1..5
    for low in (1, 0):
        p = Prog(rng, 20).init(6)
        for M in (1, 2, 3, 4, 5):
            if M == 1:
                tq = [p.act]
                mem = [('m', p.act, [low + 1]), ('m', p.act, [])]
            else:
                tq = [low] + list(range(p.act, p.act + M - 1))
                mem = [('m', t, _pick(rng, [q for q in range(p.act) if q not in tq], 2)) for t in tq] + [('d', [low + 2])]
            p.block(tq, mem)
        add(p)
    # in-place blocks with the lowest target >= 6 (k_block V = 2 / c128), 0 on a state too small for k_lowq (V = 1)
    p = Prog(rng, 14).init(14)
    for M in (1, 2, 3, 4, 5):
        tq = sorted(_pick(rng, range(6, 14), M))
        others = [q for q in range(14) if q not in tq]
        p.block(tq, [('m', t, _pick(rng, others, 3)) for t in tq] + [('d', _pick(rng, others, 2))])
    add(p)
    p = Prog(rng, 8).init(8)
    for M in (1, 2, 3, 4, 5):
        tq = [0] + sorted(_pick(rng, range(1, 8), M - 1))
        p.block(tq, [('m', t, _pick(rng, [q for q in range(8) if q not in tq], 2)) for t in tq])
    add(p)
    # k_lowq: low targets with 0, 1 and 2 high targets (LB = 9 / 8 for c64 / c128), index qubits everywhere
    LB = 9 if c64 else 8
    p = Prog(rng, 13).init(13)
    for tq in ([0, 3], [1, LB + 1], [2, LB, LB + 2], [0, 1, 2, 3, 4]):
        p.block(tq, [('m', t, _pick(rng, [q for q in range(13) if q not in tq], 3)) for t in tq] + [('d', [5, 12])])
    p.mux(0, [1, 7, 12])
    add(p)
    # diagonals: plain (and at n_active = 0), blocks with ascending runs and with descending index qubits; swaps; EXTEND
    p = Prog(rng, 12).init(0)
    p.diag([])
    p.diag_block([[], []])
    p.mux(0, [])
    p.expand(1, [[0]])
    p.swap(0, 1)
    p.extend(5)
    p.mux(2, [0, 1])
    p.swap(1, 3)
    p.diag([4, 0, 2])
    p.diag_block([[0, 1, 2], [3, 4], [1]])
    p.diag_block([[3, 0], [2, 1]])
    p.extend(9)
    add(p)
    return out


def random_lazy_program(rng, n_local, n_ops=10, global_q=()):
    """A seeded random program over the lazily materialised schedule: INIT over n0 < n_local, expansions of 1..8
    qubits, in-place blocks of 1..5 targets at any height, diagonals and diagonal blocks, swaps, EXTEND; index qubits
    drawn from the materialised ones and from `global_q`."""
    p = Prog(rng, n_local).init(int(rng.randint(0, max(1, n_local - 3))))
    for _ in range(n_ops):
        k = rng.randint(7)
        room = n_local - p.act
        pool = list(range(p.act)) + list(global_q)
        if k <= 1 and room >= 1:
            M = int(rng.randint(1, min(8, room) + 1))
            if M > 5:
                p.expand(M, [_pick(rng, pool, int(rng.randint(0, 3))) for _ in range(M)], n_diag=int(rng.randint(0, 3)),
                         diag_ctrl=_pick(rng, pool, 2))
            else:
                p.expand(M, [_pick(rng, pool, int(rng.randint(0, 4))) for _ in range(M)], n_diag=int(rng.randint(0, 2)),
                         diag_ctrl=_pick(rng, pool, 3))
        elif k == 2 and p.act >= 2:
            M = int(rng.randint(1, min(5, p.act - 1) + 1))
            tq = sorted(_pick(rng, range(p.act), M))
            others = [q for q in pool if q not in tq]
            mem = [('m', tq[int(rng.randint(M))], _pick(rng, others, int(rng.randint(0, 4)))) for _ in range(int(rng.randint(1, 7)))]
            if rng.rand() < 0.4:
                mem.insert(int(rng.randint(len(mem) + 1)), ('d', _pick(rng, others, 2)))
            p.block(tq, mem)
        elif k == 3 and p.act >= 1:
            t = int(rng.randint(p.act))
            p.mux(t, _pick(rng, [q for q in pool if q != t], int(rng.randint(0, 4))))
        elif k == 4:
            cs = [sorted(_pick(rng, pool, int(rng.randint(0, 4)))) for _ in range(int(rng.randint(1, 4)))]
            if rng.rand() < 0.3:
                cs[0] = cs[0][::-1]
            p.diag_block(cs) if len(cs) > 1 else p.diag(cs[0])
        elif k == 5 and p.act >= 2:
            a, b = _pick(rng, range(p.act), 2)
            p.swap(a, b)
        elif room >= 1:
            p.extend(p.act + int(rng.randint(1, room + 1)))
    return p.finish() + (p.act,)


def _run_and_compare(h, ops, tabs, n, precision, n_global=0, rank=0, what=''):
    want, act = em.run_plan(_plan(ops, tabs, n), n_global=n_global, rank=rank)
    h.run_program(ops, tabs)
    got = h.get_amplitudes().astype(np.complex128)
    assert h.get_active() == act, what
    err = np.abs(got - want).max()
    assert err < TOL_AMP[precision], (what, err)
    return want, act


# ---- (1) + (2a) census and plain handles --------------------------------------------------------------------
@pytest.mark.parametrize('precision', ['double', 'single'])
def test_kernel_census_and_plain_handles(precision):
    """The census corpus on plain handles: amplitudes against the op semantics (never-materialised memory holds
    NaN and must never be read), and the union of the recorded kernels is exactly the declared list."""
    seen = set()
    for i, (n, ops, tabs) in enumerate(census_corpus(precision)):
        with _native.Handle(n, precision) as h:
            h.set_amplitudes(np.full(1 << n, np.nan + 1j * np.nan), 0, n_active=0)
            _run_and_compare(h, ops, tabs, n, precision, what=('census', i))
            seen |= set(h.op_kernels())
    want = census_names(precision)
    assert seen == want, ('missing', sorted(want - seen), 'unexpected', sorted(seen - want))


@pytest.mark.parametrize('precision', ['double', 'single'])
def test_random_lazy_programs_on_plain_handles(precision):
    rng = np.random.RandomState(600 if precision == 'double' else 601)
    for trial in range(40):
        n = int(rng.randint(1, 18))
        ops, tabs, _ = random_lazy_program(rng, n, int(rng.randint(3, 12)))
        with _native.Handle(n, precision) as h:
            h.set_amplitudes(np.full(1 << n, np.nan + 1j * np.nan), 0, n_active=0)
            _run_and_compare(h, ops, tabs, n, precision, what=('random', trial))


@pytest.mark.parametrize('precision', ['double', 'single'])
def test_refusals_are_errors_not_wrong_states(precision):
    """Blocks the engine cannot serve come back as QCM_ERR_UNSUPPORTED: a wide expansion with more than four
    diagonal members, and member tables over 160 KiB of shared memory."""
    rng = np.random.RandomState(3)
    p = Prog(rng, 12).init(4)
    p.expand(6, [[0]] * 6, n_diag=5, diag_ctrl=[1])
    with _native.Handle(12, precision) as h:
        with pytest.raises(_native.NativeError) as ei:
            h.run_program(*p.finish())
        assert ei.value.code == -4
    p = Prog(rng, 14).init(14)
    p.block([12, 13], [('m', 12 + (g % 2), list(range(10))) for g in range(F.QCM_MAX_MEMBERS)])
    with _native.Handle(14, precision) as h:
        with pytest.raises(_native.NativeError) as ei:
            h.run_program(*p.finish())
        assert ei.value.code == -4


# ---- (2b) index qubits at 31 .. 61: a sharded handle's global qubits --------------------------------------------
GLOBAL_Q = (31, 32, 33, 47, 61)


@pytest.mark.parametrize('precision', ['double', 'single'])
@pytest.mark.parametrize('n_local', [10, 14])
def test_global_index_qubits(precision, n_local):
    """Index qubits at 31, 32, 33, 47 and 61 of a handle sharded over 62 - n_local global qubits: every kernel's 64-bit
    index branch and rank_bits.  The rank's bits differ across those qubits; post-selection masks include them."""
    n_global = 62 - n_local
    gq = [q for q in GLOBAL_Q if q >= n_local]
    rng = np.random.RandomState(700 + n_local)
    ranks = [sum(((k >> j) & 1) << (q - n_local) for j, q in enumerate(gq)) for k in (0b10110, 0b01001)]
    idx = np.arange(1 << n_local, dtype=np.int64)
    for rank in ranks:
        with _native.Handle(n_local, precision) as h:
            h.set_shard(n_global, rank)
            progs = []
            # every path with a global index qubit: expansions (table, tree, Q0), blocks at both heights, k_lowq,
            # diagonals, diagonal blocks, a plain MUX1Q
            p = Prog(rng, n_local).init(3)
            p.expand(2, [[gq[0], 0], [gq[-1]]])
            p.expand(4, [[gq[1]], [gq[2], 1], [], [gq[3]]], n_diag=1, diag_ctrl=[gq[4], 2])
            p.block([0, 2], [('m', 0, [gq[0], 5]), ('m', 2, [gq[4], gq[1], 1]), ('d', [gq[2], 3])])
            p.expand(min(4, n_local - p.act), [[gq[3], 4], [gq[2]], [gq[1]], [gq[0]]][:min(4, n_local - p.act)])
            progs.append(p.finish())
            p = Prog(rng, n_local).init(n_local)
            p.block([0, 3], [('m', 0, [gq[4], 5]), ('m', 3, [gq[0], gq[1]])])
            p.block([n_local - 2, n_local - 1], [('m', n_local - 1, [gq[2], 0]), ('m', n_local - 2, [gq[3]])])
            p.mux(1, [gq[1], gq[4], 0])
            p.diag([gq[0], 2, gq[4]])
            p.diag_block([[0, 1, gq[0]], [gq[1], gq[2], gq[3]], [gq[4]]])
            p.diag_block([[gq[4], 3], [gq[0], 1]])
            progs.append(p.finish())
            p = Prog(rng, n_local).init(1)
            p.expand(n_local - 1 if n_local - 1 <= 8 else 8, [[gq[j % len(gq)], 0] for j in range(min(8, n_local - 1))])
            progs.append(p.finish())
            for _ in range(6):
                ops, tabs, _a = random_lazy_program(rng, n_local, 8, global_q=gq)
                progs.append((ops, tabs))
            for k, (ops, tabs) in enumerate(progs):
                want, act = _run_and_compare(h, ops, tabs, n_local, precision, n_global, rank, ('global', rank, k))
                w = np.abs(want) ** 2
                gi = idx | (rank << n_local)
                # post-selection masks that include global bits (value matching and not matching the rank) and local ones
                for mask, value, nb in (((1 << gq[0]) | (1 << gq[3]) | 1, (rank << n_local) & ((1 << gq[0]) | (1 << gq[3])), 4),
                                        ((1 << gq[1]) | (1 << (act - 1 if act else 0)), (1 << gq[1]) & (rank << n_local), min(3, act)),
                                        ((1 << gq[2]), ((rank << n_local) & (1 << gq[2])) ^ (1 << gq[2]), 2)):
                    probs, kept = h.postselect(mask, value, nb)
                    sel = (gi & mask) == value
                    ref = np.zeros(1 << nb)
                    np.add.at(ref, idx[sel] & ((1 << nb) - 1), w[sel])
                    assert abs(kept - w[sel].sum()) <= TOL_REL[precision] * max(w.sum(), 1e-300), (k, mask)
                    assert np.allclose(probs, ref, rtol=TOL_REL[precision], atol=1e-15 if precision == 'double' else 1e-7), (k, mask)


# ---- (2c) batched handles on the lazy corpus ---------------------------------------------------------------------
@pytest.mark.parametrize('precision', ['double', 'single'])
def test_batched_lazy_programs(precision):
    """B = 3..5 states with per-point tables (the expansion kernels' btab / btab64 / bctab strides, k_diag_multi, the
    tree and the post-selection at n_active < n_local with the n_local batch stride)."""
    rng = np.random.RandomState(800 if precision == 'double' else 801)
    for trial in range(10):
        n = int(rng.randint(4, 15))
        B = int(rng.randint(3, 6))
        ops, tabs, act = random_lazy_program(rng, n, int(rng.randint(3, 10)))
        if act < 3:
            continue
        rows = [tabs] + [tabs * (1.0 + 0.3 * rng.standard_normal(tabs.shape)) for _ in range(B - 1)]
        with _native.Handle(n, precision, batch=B) as h:
            h.run_program(ops, np.stack(rows))
            assert h.get_active() == act
            wants = []
            for y in range(B):
                want, a2 = em.run_plan(_plan(ops, rows[y], n))
                h.batch_select(y)
                got = h.get_amplitudes().astype(np.complex128)
                scale = max(np.abs(want).max(), 1e-30)
                assert np.abs(got - want).max() / scale < (1e-11 if precision == 'double' else 2e-5), (trial, y)
                wants.append(np.abs(want) ** 2)
            mask = 1 << (act - 1)
            nb = act - 2
            probs, kept = h.postselect(mask, 0, nb)
            kept2 = h.postselect_resident(mask, 0, nb)
            assert np.array_equal(kept, kept2)
            S = 4000
            keys = h.sample_batched(S, 17, np.arange(B) + 40)
            again = h.sample_batched(S, 17, np.arange(B) + 40)
            assert np.array_equal(keys, again)
            idx = np.arange(1 << n)
            for y in range(B):
                w = wants[y]
                sel = (idx & mask) == 0
                ref = np.zeros(1 << nb)
                np.add.at(ref, idx[sel] & ((1 << nb) - 1), w[sel])
                tol = 1e-9 if precision == 'double' else 2e-4
                assert abs(kept[y] - w[sel].sum()) <= tol * w.sum(), (trial, y)
                assert np.allclose(probs[y], ref, rtol=tol, atol=tol * w.sum() * 1e-3), (trial, y)
                assert np.array_equal(h.fetch_probs(y, nb), probs[y])
                k = keys[y].astype(np.int64)
                assert k.max() < (1 << act) and (w[k] > 0).all()
                marg = np.bincount(k >> (act - 3), minlength=8) / S
                wm = np.bincount(idx >> (act - 3), weights=w, minlength=1 << (n - act + 3))[:8] / w.sum()
                assert 0.5 * np.abs(marg - wm).sum() < weissman_tv_bound(8, S, 1e-7)


# ---- (3) the small-circuit kernel ------------------------------------------------------------------------------
def _small_program(rng, N):
    """Fully materialised program over N qubits with every op k_small interprets."""
    p = Prog(rng, N)
    if N == 0 or rng.rand() < 0.8:
        p.init(N)
    else:
        p.act = N                               # no INIT: the kernel starts from |0..0>
    for _ in range(int(rng.randint(0, 10)) if N else 0):
        k = rng.randint(5)
        if k == 0:
            t = int(rng.randint(N))
            p.mux(t, _pick(rng, [q for q in range(N) if q != t], int(rng.randint(0, min(N - 1, 4) + 1))))
        elif k == 1:
            p.diag(_pick(rng, range(N), int(rng.randint(0, min(N, 5) + 1))))
        elif k == 2 and N >= 2:
            p.swap(*_pick(rng, range(N), 2))
        elif k == 3 and N >= 2:
            M = int(rng.randint(1, min(5, N - 1) + 1))
            tq = sorted(_pick(rng, range(N), M))
            others = [q for q in range(N) if q not in tq]
            mem = [('m', tq[int(rng.randint(M))], _pick(rng, others, int(rng.randint(0, 3)))) for _ in range(int(rng.randint(1, 5)))]
            mem.insert(int(rng.randint(len(mem) + 1)), ('d', _pick(rng, others, 2)))
            p.block(tq, mem)
        elif k == 4:
            p.diag_block([_pick(rng, range(N), int(rng.randint(0, 4))) for _ in range(2)])
    return p.finish()


@pytest.mark.parametrize('precision', ['double', 'single'])
def test_small_kernel_fuzz(precision):
    """_native.run_batch_small on one batch of random programs of 0..13 qubits (shared memory sized by the largest):
    pmf and kept mass against the op semantics, shots against the exact key distribution, determinism per
    (seed, stream), and the same programs on a Handle."""
    rng = np.random.RandomState(900 if precision == 'double' else 901)
    plans, cmaps, ps, ws = [], [], [], []
    for c in range(60):
        N = c % 14
        ops, tabs = _small_program(rng, N)
        pl = _plan(ops, tabs, N)
        plans.append(pl)
        full = np.zeros(1 << N, dtype=np.complex128)
        if len(ops) and int(ops[0]['kind']) == F.QCM_OP_INIT_PRODUCT:
            want, _ = em.run_plan(pl)
        else:
            e0 = F._Emitter()
            e0.op(F.QCM_OP_INIT_PRODUCT, n_in=0, n_out=N, table_off=e0.table(np.tile([1.0, 0, 0, 0], (max(N, 1), 1))))
            o0, t0 = e0.finish()
            o = np.concatenate([o0, ops.copy()])
            o['table_off'][1:] += t0.size
            want, _ = em.run_plan(_plan(o, np.concatenate([t0, tabs]), N))
        full[:] = want
        ws.append(np.abs(full) ** 2)
        ncl = int(rng.randint(0, min(N, 6) + 2)) if N else 0
        cm = np.array([int(rng.randint(-1, N)) for _ in range(ncl)], dtype=np.int32)
        cmaps.append(cm)
        bits = int(rng.randint(0, N + 1))
        mask = int(rng.randint(0, 1 << N)) if N else 0
        value = mask & int(rng.randint(0, 1 << N)) if N else 0
        ps.append((mask, value, bits))
    sids = rng.permutation(1000)[:len(plans)]
    S = 20000
    keys, probs, kept, _ms = _native.run_batch_small(plans, cmaps, ps, S, 77, precision=precision, stream_ids=sids)
    keys2, _p, _k, _ = _native.run_batch_small(plans, cmaps, ps, S, 77, precision=precision, stream_ids=sids)
    assert np.array_equal(keys, keys2)
    for c, (pl, cm, (mask, value, bits), w) in enumerate(zip(plans, cmaps, ps, ws)):
        N = pl.n_phys
        idx = np.arange(1 << N)
        sel = (idx & mask) == value
        ref = np.zeros(1 << bits)
        np.add.at(ref, idx[sel] & ((1 << bits) - 1), w[sel])
        if precision == 'double':
            assert abs(kept[c] - w[sel].sum()) < 1e-12 and np.abs(probs[c] - ref).max() < 1e-12, c
        else:
            assert abs(kept[c] - w[sel].sum()) <= 2e-4 * max(w[sel].sum(), 1e-3), c
            assert np.abs(probs[c] - ref).max() <= 2e-4 * max(ref.max(), 1e-3), c
        # key distribution: clbit j <- qubit cm[j] (-1: always 0)
        key = np.zeros(1 << N, dtype=np.int64) if len(cm) else idx.copy()       # no clbit map: raw basis-state keys
        for j, q in enumerate(cm):
            if q >= 0:
                key |= ((idx >> int(q)) & 1) << j
        K = 1 << len(cm) if len(cm) else 1 << N
        kp = np.bincount(key, weights=w, minlength=K)
        obs = np.bincount(keys[c].astype(np.int64), minlength=K) / S
        assert len(obs) == K and (obs[kp < 1e-14] == 0).all(), c
        assert 0.5 * np.abs(obs - kp / kp.sum()).sum() < weissman_tv_bound(K, S, 1e-8), c
    # the same programs on a Handle (INIT-started ones): the pmfs agree
    for c, (pl, (mask, value, bits)) in enumerate(zip(plans, ps)):
        if pl.n_phys == 0 or not len(pl.ops) or int(pl.ops[0]['kind']) != F.QCM_OP_INIT_PRODUCT:
            continue
        with _native.Handle(pl.n_phys, precision) as h:
            h.run_program(pl.ops, pl.tables)
            p2, k2 = h.postselect(mask, value, bits)
        tol = 1e-12 if precision == 'double' else 2e-4
        assert np.abs(p2 - probs[c]).max() <= tol * max(1.0, probs[c].max()) and abs(k2 - kept[c]) <= tol, c


@pytest.mark.parametrize('seed', range(2))
def test_random_generic_circuits_on_the_engine(seed):
    """Random foreign circuits through B200Simulator.run on the real engine, small and large path: the
    post-selected pmf and success probability against a textbook simulation, keys in the support."""
    from test_host_fusion import _random_circuit, _textbook_state
    from qcmrf_b200 import B200Simulator, transpile
    from qcmrf_b200.circuit import QuantumCircuit
    rng = np.random.RandomState(9300 + seed)
    sims = [B200Simulator(precision='double', small_batch=s, seed=1) for s in (True, False)]
    for trial in range(10):
        nq = int(rng.randint(1, 9))
        base = _random_circuit(rng, nq, int(rng.randint(1, 30)))
        pw = np.abs(_textbook_state(base)) ** 2
        nv = int(rng.randint(1, nq + 1))
        c = QuantumCircuit(nq, nq)
        for ins in base.data:
            c._qc_add(ins.operation, list(ins.qubits))
        c.measure(range(nq), range(nq))
        if trial % 2:
            c = transpile(c, basis_gates=['cx', 'id', 'rz', 'sx', 'x'])
        kept = pw[:1 << nv].sum()
        if kept < 1e-9:
            continue
        for sim in sims:
            res = sim.run(c, shots=2000, n_vars=nv).result()
            p, d = res.postselected_probabilities(0)
            assert np.abs(p - pw[:1 << nv] / kept).max() < 1e-10 and abs(d - kept) < 1e-10, (seed, trial, sim.small_batch)
            cnt = res.get_counts()
            assert sum(cnt.values()) == 2000 and all(pw[int(k, 2)] > 1e-14 for k in cnt)
    for s in sims:
        s.close()


# ---- (4) states past 2^31 and 2^32 amplitudes ------------------------------------------------------------------
def _free_gpu_bytes():
    try:
        import torch
        return torch.cuda.mem_get_info()[0]
    except Exception:
        return 0


@pytest.mark.parametrize('precision,n_local', [('single', 32), ('double', 31), ('single', 33)])
def test_states_past_2_to_31_amplitudes(precision, n_local):
    """SLOW PART (32 / 64 GiB states).  A product state over n_local - 1 qubits, the top qubit materialised by an
    expansion whose writes cross index 2^31 (2^32 for 33 qubits), then blocks (low and high targets), k_lowq, a
    diagonal, a diagonal block and a swap -- all inside T = {0..5} plus the top three qubits.  The state factorises
    into (product over the spectator qubits) x (a 2^9 state on T), which numpy computes exactly."""
    need = (8 if precision == 'single' else 16) << n_local
    if _free_gpu_bytes() < need + (8 << 30):
        pytest.skip('needs %d GiB of free device memory' % ((need >> 30) + 8))
    rng = np.random.RandomState(n_local)
    top = n_local - 1
    T = [0, 1, 2, 3, 4, 5, top - 2, top - 1, top]
    tpos = {q: j for j, q in enumerate(T)}
    v = rng.randn(n_local - 1, 2) + 1j * rng.randn(n_local - 1, 2)
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    qv = np.stack([v[:, 0].real, v[:, 0].imag, v[:, 1].real, v[:, 1].imag], axis=1)

    def build(n, q, init_rows):
        """The program with qubit labels q(.) on n stored qubits; table draws do not depend on the labels."""
        p = Prog(np.random.RandomState(99), n).init(n - 1, init_rows)
        tp = n - 1
        p.mux(tp, [q(0), q(top - 1)])
        p.block([q(0), q(2)], [('m', q(0), [tp, q(1)]), ('m', q(2), [q(top - 2)]), ('d', [tp, q(4)])])   # k_lowq
        p.block([q(top - 1), tp], [('m', tp, [q(3)]), ('m', q(top - 1), [q(0), q(5)])])               # k_block, high targets
        p.diag([tp, q(1), q(top - 2)])
        p.diag_block([[q(0), q(1), q(2)], [q(top - 1), tp]])
        p.swap(q(3), q(top - 1))
        return p.finish()
    ops, tabs = build(n_local, lambda x: x, qv)
    small, stabs = build(len(T), lambda x: tpos[x], qv[T[:-1]])
    phiT, _ = em.run_plan(_plan(small, stabs, len(T)))
    spect = [q for q in range(n_local - 1) if q not in tpos]

    def amp(i):
        i = np.asarray(i, dtype=np.int64)
        t = np.zeros_like(i)
        for q, j in tpos.items():
            t |= ((i >> q) & 1) << j
        a = phiT[t]
        for q in spect:
            a = a * v[q, (i >> q) & 1]
        return a

    with _native.Handle(n_local, precision) as h:
        h.run_program(ops, tabs)
        kn = h.op_kernels()
        assert kn[1].startswith('k_expand<') and kn[2].startswith('k_lowq') and kn[3].startswith('k_block<'), kn
        tol = TOL_AMP[precision]
        edges = [0, 1 << 30, 1 << 31, (1 << n_local) - 1024] + ([1 << 32] if n_local > 32 else [])
        firsts = [max(0, min(e - 512, (1 << n_local) - 1024)) for e in edges]
        firsts += [int(x) & ~1023 for x in rng.randint(0, 1 << (n_local - 10), 58) << 10]
        for f in firsts:
            got = h.get_amplitudes(f, 1024).astype(np.complex128)
            assert np.abs(got - amp(np.arange(f, f + 1024))).max() < tol, f
        # post-selection: the spectators' mass is 1, so masses over T are exact
        wT = np.abs(phiT) ** 2
        tidx = np.arange(1 << len(T))
        for mask, value in (((1 << top) | (1 << (top - 1)), 0), ((1 << top) | (1 << 4), 1 << top)):
            probs, kept = h.postselect(mask, value, 6)
            tm = sum(1 << tpos[q] for q in T if (mask >> q) & 1)
            tv = sum(1 << tpos[q] for q in T if (value >> q) & 1)
            sel = (tidx & tm) == tv
            ref = np.bincount(tidx[sel] & 63, weights=wT[sel], minlength=64)
            assert abs(kept - wT[sel].sum()) <= TOL_REL[precision] * 4, (mask, kept, wT[sel].sum())
            # the product factor of qubits 0..5 is part of phiT; spectators sum to one
            assert np.allclose(probs, ref, rtol=TOL_REL[precision] * 4, atol=1e-9)
        S = 200000
        keys = h.sample(S, 5, 1).astype(np.int64)
        assert (np.abs(amp(keys)) > 0).all()
        assert (keys >= (1 << top)).any()                 # the materialised top qubit: past 2^31 (c64 32, 33)
        t = np.zeros_like(keys)
        for q, j in tpos.items():
            t |= ((keys >> q) & 1) << j
        obs = np.bincount(t, minlength=1 << len(T)) / S
        assert 0.5 * np.abs(obs - wT / wT.sum()).sum() < weissman_tv_bound(1 << len(T), S)


# ---- (5) launch knobs, one child process each -------------------------------------------------------------------
#: knob -> does it leave every amplitude bit-identical to the default?  (Tile order, thread count, grid size and
#: resident CTAs do not change any amplitude's arithmetic; the rotated-pass shape, k_block in place of k_lowq and
#: the unrotated last pass compute the same values by other instruction sequences.)
KNOBS = [({'QCM_LOW_SHAPE': '8x10'}, False), ({'QCM_LOW_SHAPE': '4x7'}, False), ({'QCM_LOW_SHAPE': '2x6'}, False),
         ({'QCM_LOW_SHAPE': '1x5'}, False), ({'QCM_LOW_CTAS': '1'}, True), ({'QCM_LOW_CTAS': '0'}, True),
         ({'QCM_EXPAND_SCHED': 'counter'}, True), ({'QCM_EXPAND_THREADS': '64'}, True), ({'QCM_EXPAND_THREADS': '1024'}, True),
         ({'QCM_GRID_MULT': '1'}, True), ({'QCM_LOWQ': '0'}, False), ({'QCM_ROTATE': '0'}, False),
         ({'QCM_PRODUCT_SAMPLE': '0'}, True)]

# QCM_GRID_MULT=1 caps a streaming grid at 148 SMs x (at most 8 resident CTAs of 256 threads): k_block with M <= 2
# in complex64 covers 2^(N-2) / U vectors per ... 256 * U per CTA, i.e. 2^(N-12) CTAs; N = 23 needs 2048 > 148 * 8.
GRID_N = 23
assert (1 << (GRID_N - 12)) > 148 * 8


def _knob_corpus():
    progs = []
    for precision in ('single', 'double'):
        for n, ops, tabs in census_corpus(precision, seed=5):
            progs.append((precision, n, ops, tabs))
    rng = np.random.RandomState(21)
    p = Prog(rng, GRID_N).init(GRID_N - 2)
    p.expand(2, [[0, 3], [GRID_N - 3]])
    p.block([7], [('m', 7, [0, GRID_N - 1])])
    p.block([8, GRID_N - 1], [('m', 8, [1]), ('m', GRID_N - 1, [2])])
    p.diag([0, GRID_N - 1])
    p.swap(2, GRID_N - 2)
    ops, tabs = p.finish()
    progs.append(('single', GRID_N, ops, tabs))
    return progs


def _knob_child(out_path):
    """Run the knob corpus in this process (the knobs are read once per process) and store the results."""
    res = {}
    for k, (precision, n, ops, tabs) in enumerate(_knob_corpus()):
        with _native.Handle(n, precision) as h:
            h.run_program(ops, tabs)
            res['amp%d' % k] = h.get_amplitudes()
            res['kern%d' % k] = np.array(h.op_kernels())
            if k % 4 == 0 or n == GRID_N:
                res['keys%d' % k] = h.sample(20000, 3, 1)
    # a product state (sampled qubit by qubit unless QCM_PRODUCT_SAMPLE=0)
    rng = np.random.RandomState(4)
    p = Prog(rng, 10).init(10)
    ops, tabs = p.finish()
    with _native.Handle(10, 'double') as h:
        h.run_program(ops, tabs)
        res['prod_keys'] = h.sample(100000, 9, 2)
        res['prod_amp'] = h.get_amplitudes()
    np.savez(out_path, **res)


def _spawn(tmp_path, name, env_extra):
    out = str(tmp_path / ('%s.npz' % name))
    env = dict(os.environ)
    for k in [k for k in env if k.startswith('QCM_')]:
        del env[k]
    env.update(env_extra)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), out], env=env, timeout=600, capture_output=True, text=True)
    assert r.returncode == 0, (env_extra, r.stdout[-2000:], r.stderr[-2000:])
    return dict(np.load(out))


def test_launch_knobs_in_child_processes(tmp_path):
    corpus = _knob_corpus()
    refs = [em.run_plan(_plan(ops, tabs, n))[0] for precision, n, ops, tabs in corpus]
    base = _spawn(tmp_path, 'default', {})
    for env_extra, identical in [({}, True)] + KNOBS:
        got = base if not env_extra else _spawn(tmp_path, '_'.join('%s=%s' % kv for kv in env_extra.items()), env_extra)
        for k, (precision, n, ops, tabs) in enumerate(corpus):
            a = got['amp%d' % k].astype(np.complex128)
            assert np.abs(a - refs[k]).max() < TOL_AMP[precision], (env_extra, k)
            if identical:
                assert np.array_equal(got['amp%d' % k], base['amp%d' % k]), (env_extra, k)
            if 'keys%d' % k in got:
                w = np.abs(refs[k]) ** 2
                keys = got['keys%d' % k].astype(np.int64)
                assert (w[keys] > 0).all(), (env_extra, k)
                hi = keys >> max(0, n - 6)
                obs = np.bincount(hi, minlength=64) / len(keys)
                wm = np.bincount(np.arange(1 << n) >> max(0, n - 6), weights=w, minlength=64) / w.sum()
                assert 0.5 * np.abs(obs - wm).sum() < weissman_tv_bound(64, len(keys), 1e-8), (env_extra, k)
        names = set(x for k in range(len(corpus)) for x in got['kern%d' % k])
        if 'QCM_LOW_SHAPE' in env_extra:
            w_, tb = env_extra['QCM_LOW_SHAPE'].split('x')
            assert any(x.startswith('k_expand_low<float') and x.endswith('TB=%s,NW=%s>' % (tb, w_)) for x in names), names
        if env_extra.get('QCM_LOWQ') == '0':
            assert not any(x.startswith('k_lowq') for x in names)
        if env_extra.get('QCM_ROTATE') == '0':
            assert not any(x.startswith('k_expand_low') for x in names)
        # product-state shots: the exact product law; the tree sampler draws other (equally valid) keys
        w = np.abs(got['prod_amp']) ** 2
        obs = np.bincount(got['prod_keys'].astype(np.int64), minlength=1 << 10) / len(got['prod_keys'])
        assert 0.5 * np.abs(obs - w / w.sum()).sum() < weissman_tv_bound(1 << 10, len(got['prod_keys']))
        if identical and env_extra.get('QCM_PRODUCT_SAMPLE') != '0':
            assert np.array_equal(got['prod_keys'], base['prod_keys'])


if __name__ == '__main__':
    _knob_child(sys.argv[1])
