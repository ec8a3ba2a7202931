"""State sharded over 2^g GPUs of one box: one process per GPU, torch.distributed for the
plumbing (NCCL over NVLink; gloo in the CPU tests).

Rank r holds the 2^n_local amplitudes whose g highest physical qubits spell r.  The
engine already reads index bits of global qubits from the rank (qcm_set_shard), so
controls and diagonal terms on global qubits cost nothing.  What needs care is a
gate whose *target* is global:

* a global qubit that is materialised by the op itself (known |0> on input, one
  member) needs no data from other ranks: rank r keeps the branch its own bit
  selects, i.e. the member degenerates to a diagonal factor table[idx][bit][0] that
  rides in the same sweep.  With the lazily materialised schedule every global qubit
  of a QCMRF circuit is of this kind (the last ancillas), so the whole gate program
  is communication-free; until the first global qubit materialises all ranks hold
  identical replicas of the small state.
* a global qubit that is already materialised must be brought on-GPU first: a
  qubit-swap all-to-all exchanges s global qubits with the s highest local qubits
  (contiguous slabs: rank with coordinate c sends slab j to the rank with coordinate
  j and stores what it receives as slab j).  The dense (fully materialised, one
  in-place pass per clique) schedule of SURVEY.md 8e needs exactly one such exchange
  for a QCMRF circuit; lookahead gathers every global qubit that is still going to
  be targeted into one exchange.

``shard_plan`` is pure (plan in, per-rank segments out) so its index arithmetic is
tested on the CPU for 2, 4 and 8 virtual ranks; ``ShardedSimulator`` executes the
segments on a real handle and does the collectives.
"""
import os
import time
from dataclasses import dataclass, field
from typing import List, Optional, Tuple

import numpy as np

from . import _native, fusion, ir, plancache
QCM_MAX_GATHER = 3
from .fusion import (OP_DTYPE, QCM_MAX_CTRL, QCM_OP_BLOCK, QCM_OP_DIAG, QCM_OP_EXTEND, QCM_OP_INIT_PRODUCT,
                     QCM_OP_MUX1Q, QCM_OP_SWAP, _Emitter)

__all__ = ['shard_plan', 'ShardedPlan', 'ShardedSimulator']


@dataclass
class ShardedPlan:
    g: int
    rank: int
    n_local: int
    n_phys: int
    #: ('run', ops, tables, rank_mask) | ('exchange', betas) | ('xblock', betas, ops, tables, rank_mask)
    #: -- betas: rank-bit indices, ascending
    segments: List[tuple] = field(default_factory=list)
    pos: List[int] = field(default_factory=list)      # plan-physical qubit -> final position
    mat_mask: int = 0                                  # rank bits whose global qubit is materialised at the end
    n_exchanges: int = 0
    exchange_amps: int = 0                             # amplitudes this rank sends in total


def _headers(ops):
    """Yield (index, header op, member ops) over a flat qcm_op array."""
    i = 0
    while i < len(ops):
        op = ops[i]
        if int(op['kind']) == QCM_OP_BLOCK:
            n = int(op['n_ctrl'])
            yield i, op, [ops[i + 1 + k] for k in range(n)]
            i += 1 + n
        else:
            yield i, op, ([op] if int(op['kind']) == QCM_OP_MUX1Q else [])
            i += 1


def _targets(op, members):
    k = int(op['kind'])
    if k == QCM_OP_BLOCK:
        return [int(x) for x in op['ctrl'][:int(op['target'])]]
    if k == QCM_OP_MUX1Q:
        return [int(op['target'])]
    return []


def shard_plan(pl: fusion.Plan, g: int, rank: int, fuse_exchange: bool = False) -> ShardedPlan:
    """Rewrite a single-device plan for rank ``rank`` of 2^g.  fuse_exchange: where a qubit swap is
    followed by sweeps on the swapped-in qubits, emit ONE ('xblock', ...) segment (the engine's fused
    gather pass over peer memory) instead of ('exchange', ...) plus local passes."""
    n_phys = pl.n_phys
    n_local = n_phys - g
    if n_local < 1:
        raise ValueError('state of %d qubits cannot be sharded over 2^%d ranks' % (n_phys, g))
    sp = ShardedPlan(g, rank, n_local, n_phys)
    if pl.n_global not in (0, g):
        raise ValueError('plan was laid out for %d global qubits, not %d' % (pl.n_global, g))
    if g == 0:
        sp.segments.append(('run', pl.ops, pl.tables, 0))
        sp.pos = list(range(n_phys))
        return sp
    tabs = pl.tables
    pos = list(range(n_phys))              # plan-physical qubit -> current position
    occ = list(range(n_phys))              # position -> plan-physical qubit
    mat_mask = 0                           # rank bits of materialised global qubits
    active = 0                             # plan-level n_active
    em = _Emitter()
    seg_mask = [0]

    def flush():
        if em.ops:
            ops, tb = em.finish()
            sp.segments.append(('run', ops, tb, seg_mask[0]))
        em.ops, em.tabs, em.off = [], [], 0

    def set_mask(m):
        if m != seg_mask[0]:
            flush()
            seg_mask[0] = m

    def rbit(position):
        return (rank >> (position - n_local)) & 1

    def lact(a):
        return min(a, n_local)

    headers = list(_headers(pl.ops))

    def future_targets(from_h):
        out = {}
        for hi in range(from_h, len(headers)):
            _, op, members = headers[hi]
            for t in _targets(op, members):
                out.setdefault(t, hi)
        return out

    def exchange_for(need, from_h):
        """Bring the materialised global qubits ``need`` (plan-physical) on-GPU, together with every
        other materialised global qubit that a later op targets, in one all-to-all."""
        nonlocal mat_mask
        fut = future_targets(from_h)
        cur_targets = set(_targets(headers[from_h][1], headers[from_h][2]))
        want = list(need)
        for q, _hi in sorted(fut.items(), key=lambda kv: kv[1]):
            p = pos[q]
            if q not in want and p >= n_local and (mat_mask >> (p - n_local)) & 1:
                want.append(q)
        # partners: the highest local positions whose occupants are not targeted by the current op,
        # preferring occupants that are never targeted again
        cand = [p for p in range(lact(active) - 1, -1, -1) if occ[p] not in cur_targets]
        done = [p for p in cand if occ[p] not in fut]
        s = min(len(want), len(cand))
        if s < len(need):
            raise ValueError('not enough local qubits to exchange %d global targets' % len(need))
        s = min(s, max(len(need), len(done)))
        want = want[:s]
        top = list(range(lact(active) - s, lact(active)))
        chosen = (done + [p for p in cand if p not in done])[:s]
        # make the chosen occupants sit on the top s local positions (local swaps, rarely needed)
        for tp in top:
            if tp in chosen:
                continue
            src = next(p for p in chosen if p not in top)
            chosen[chosen.index(src)] = tp
            em.op(QCM_OP_SWAP, target=src, ctrl=[tp], n_in=lact(active), n_out=lact(active))
            qa, qb = occ[src], occ[tp]
            occ[src], occ[tp] = qb, qa
            pos[qa], pos[qb] = tp, src
        flush()
        gpos = sorted(pos[q] for q in want)
        betas = [p - n_local for p in gpos]
        for gp, lp in zip(gpos, top):                 # ascending global <-> ascending top-local
            qa, qb = occ[gp], occ[lp]
            occ[gp], occ[lp] = qb, qa
            pos[qa], pos[qb] = lp, gp
        # every exchanged position stays materialised (both sides were)
        sp.n_exchanges += 1
        sp.exchange_amps += ((1 << s) - 1) << (n_local - s)
        if fuse_exchange and s <= QCM_MAX_GATHER and lact(active) == n_local:
            # sweeps that follow and only touch the swapped-in qubits ride in the same kernel
            topset = set(top)
            fused, nh = [], from_h
            while nh < len(headers):
                _, fop, fmem = headers[nh]
                if int(fop['kind']) not in (QCM_OP_MUX1Q, QCM_OP_BLOCK):
                    break
                if any(pos[t] not in topset for t in _targets(fop, fmem)):
                    break
                cand = []
                for mb in fmem:
                    ctrl = [pos[int(c)] for c in mb['ctrl'][:int(mb['n_ctrl'])]]
                    if any(c in topset for c in ctrl):
                        cand = None
                        break
                    kind = int(mb['kind'])
                    cand.append((kind, pos[int(mb['target'])] if kind == QCM_OP_MUX1Q else 0, ctrl, member_table(mb)))
                if cand is None or len(fused) + len(cand) > fusion.QCM_MAX_MEMBERS:
                    break
                fused.extend(cand)
                nh += 1
            if nh > from_h:
                xe = _Emitter()
                xe.op(QCM_OP_BLOCK, target=s, ctrl=top, n_in=n_local, n_out=n_local, n_ctrl=len(fused))
                for k, t, c, tab in fused:
                    xe.op(k, target=t, ctrl=c, n_in=n_local, n_out=n_local, table_off=xe.table(tab))
                xops, xtabs = xe.finish()
                sp.segments.append(('xblock', betas, xops, xtabs, mat_mask))
                return nh
        sp.segments.append(('exchange', betas))
        return None

    def force_materialise(position):
        """Global qubit known |0> becomes an explicit sharded qubit: ranks whose bit is 1 hold zeros."""
        nonlocal mat_mask
        if rbit(position):
            em.op(QCM_OP_DIAG, ctrl=[], n_in=lact(active), n_out=lact(active), table_off=em.table(np.zeros(2)))
        mat_mask |= 1 << (position - n_local)

    def member_table(mb):
        nc = int(mb['n_ctrl'])
        per = 2 if int(mb['kind']) == QCM_OP_DIAG else 8
        o = int(mb['table_off'])
        return tabs[o:o + (per << nc)]

    skip_to = 0
    for hi, (_, op, members) in enumerate(headers):
        if hi < skip_to:
            continue
        kind = int(op['kind'])
        n_in, n_out = int(op['n_active_in']), int(op['n_active_out'])
        if kind == QCM_OP_INIT_PRODUCT:
            set_mask(mat_mask)
            qv = tabs[int(op['table_off']):int(op['table_off']) + 4 * max(n_out, 1)].reshape(-1, 4).copy()
            scale = 1.0 + 0j
            if pl.n_global:
                # control-only qubits on the global positions: this rank holds the branch its bits select
                f = 1.0 + 0j
                for p, v in pl.global_init.items():
                    f *= complex(v[rbit(p)])
                    mat_mask |= 1 << (p - n_local)
                v0 = complex(qv[0, 0], qv[0, 1]) * f
                v1 = complex(qv[0, 2], qv[0, 3]) * f
                qv[0] = [v0.real, v0.imag, v1.real, v1.imag]
                scale = f
            elif n_out > n_local:
                f = 1.0 + 0j
                for p in range(n_local, n_out):
                    b = rbit(p)
                    f *= complex(qv[p, 2 * b], qv[p, 2 * b + 1])
                    mat_mask |= 1 << (p - n_local)
                v0 = complex(qv[0, 0], qv[0, 1]) * f
                v1 = complex(qv[0, 2], qv[0, 3]) * f
                qv = qv[:n_local].copy()
                qv[0] = [v0.real, v0.imag, v1.real, v1.imag]
            em.op(QCM_OP_INIT_PRODUCT, n_in=0, n_out=lact(n_out), table_off=em.table(qv))
            if lact(n_out) == 0 and scale != 1.0:
                # no local product qubit to carry the branch amplitude: scale the single amplitude
                em.op(QCM_OP_DIAG, ctrl=[], n_in=0, n_out=0, table_off=em.table(np.array([scale.real, scale.imag])))
            active = n_out
            set_mask(mat_mask)
            continue
        if kind == QCM_OP_EXTEND:
            set_mask(mat_mask)
            if lact(n_out) > lact(n_in):
                em.op(QCM_OP_EXTEND, n_in=lact(n_in), n_out=lact(n_out))
            active = max(active, min(n_out, n_local))
            for p in range(max(n_in, n_local), n_out):
                force_materialise(p)
            active = n_out
            set_mask(mat_mask)
            continue
        if kind == QCM_OP_SWAP:
            a, b = pos[int(op['target'])], pos[int(op['ctrl'][0])]
            if a >= n_local or b >= n_local:
                raise NotImplementedError('SWAP on a global qubit')
            set_mask(mat_mask)
            em.op(QCM_OP_SWAP, target=a, ctrl=[b], n_in=lact(active), n_out=lact(active))
            continue
        if kind == QCM_OP_DIAG:
            set_mask(mat_mask)
            ctrl = [pos[int(c)] for c in op['ctrl'][:int(op['n_ctrl'])]]
            em.op(QCM_OP_DIAG, ctrl=ctrl, n_in=lact(active), n_out=lact(active), table_off=em.table(member_table(op)))
            continue
        # ---- MUX1Q / BLOCK ---------------------------------------------------------------
        tq = _targets(op, members)
        per_target = {t: 0 for t in tq}
        for mb in members:
            if int(mb['kind']) == QCM_OP_MUX1Q:
                per_target[int(mb['target'])] += 1
        set_mask(mat_mask)
        new_global = [t for t in tq if t >= n_in and pos[t] >= n_local]
        branch = {}                                       # target -> this rank's bit (diag rewrite)
        for t in new_global:
            if per_target[t] == 1:
                branch[t] = rbit(pos[t])
            else:
                force_materialise(pos[t])
        old_global = [t for t in tq if t not in branch and pos[t] >= n_local]
        if old_global:
            # new local qubits of this op are not materialised yet; exchange among materialised ones
            nxt = exchange_for(old_global, hi)
            set_mask(mat_mask)
            if nxt is not None:                       # this op (and maybe more) went into the fused gather pass
                skip_to = nxt
                continue
        local_t = sorted(pos[t] for t in tq if t not in branch)
        l_in = lact(n_in)
        l_out = max([l_in] + [p + 1 for p in local_t])
        out_members = []
        for mb in members:
            nc = int(mb['n_ctrl'])
            ctrl = [pos[int(c)] for c in mb['ctrl'][:nc]]
            tab = member_table(mb)
            if int(mb['kind']) == QCM_OP_DIAG:
                out_members.append((QCM_OP_DIAG, 0, ctrl, tab))
                continue
            t = int(mb['target'])
            if t in branch:
                m = tab.reshape(-1, 8)
                b = branch[t]
                out_members.append((QCM_OP_DIAG, 0, ctrl, np.ascontiguousarray(m[:, 4 * b:4 * b + 2])))
            else:
                out_members.append((QCM_OP_MUX1Q, pos[t], ctrl, tab))
        flags = int(op['flags'])
        if not local_t:
            # every target was a new global qubit: only diagonal factors remain -- merge them
            for d in _merge_diags(out_members):
                em.op(QCM_OP_DIAG, ctrl=d[0], n_in=l_in, n_out=l_in, table_off=em.table(d[1]))
        elif len(out_members) == 1 and out_members[0][0] == QCM_OP_MUX1Q:
            k, t, c, tab = out_members[0]
            em.op(QCM_OP_MUX1Q, target=t, ctrl=c, n_in=l_in, n_out=l_out, table_off=em.table(tab))
            em.ops[-1]['flags'] = flags
        else:
            em.op(QCM_OP_BLOCK, target=len(local_t), ctrl=local_t, n_in=l_in, n_out=l_out, n_ctrl=len(out_members))
            em.ops[-1]['flags'] = flags
            for k, t, c, tab in out_members:
                em.op(k, target=t, ctrl=c, n_in=l_in, n_out=l_out, table_off=em.table(tab))
        for t in branch:
            mat_mask |= 1 << (pos[t] - n_local)
        active = max(active, n_out)
        set_mask(mat_mask)
    flush()
    sp.pos = pos
    sp.mat_mask = mat_mask
    return sp


def _merge_diags(members):
    """[(kind, target, ctrl, table (2^m, 2) float64)] of diagonal members -> merged [(ctrl, table (2^m, 2))]."""
    items = []
    for k, _t, ctrl, tab in members:
        assert k == QCM_OP_DIAG
        d = tab.reshape(-1, 2)
        items.append((ctrl, d[:, 0] + 1j * d[:, 1]))
    return [(c, np.stack([t.real, t.imag], axis=1)) for c, t in fusion.merge_diagonals(items)]


# ------------------------------------------------------------------------------------------
def plan_for_shards(fc, g, rank, lazy, block_max, n_global, expand_max, fuse_exchange):
    """(plan, this rank's ShardedPlan).  The lazily materialised layout is used where it is communication-free (every
    QCMRF circuit: ancillas are materialised where they live).  A circuit that would need a qubit-swap exchange in the
    middle of a lazily materialised program -- a foreign circuit that targets its high qubits again and again -- is
    planned densely instead (every qubit materialised up front, one pass per sweep, Aer's width): exchanges of partially
    materialised shards and rank-dependent pruning around them are where a seeded fuzz of random circuits on 4 ranks
    found ranks disagreeing on the segment list.  The decision looks at every rank's rewrite, so all ranks take it
    alike."""
    def build(lz):
        p = fusion.plan(fc, lazy=lz, block_max=block_max, n_global=n_global if lz else 0, expand_max=expand_max)
        return p, shard_plan(p, g, rank, fuse_exchange=fuse_exchange)
    try:
        p, q = build(lazy)
        dense = bool(lazy and g and any(shard_plan(p, g, r, fuse_exchange=fuse_exchange).n_exchanges for r in range(1 << g)))
    except ValueError:
        if not lazy:
            raise
        dense = True                                         # e.g. too few local qubits for a lazy plan's exchange
    if dense:
        p, q = build(False)
    return p, q


class _ShardPrepared:
    __slots__ = ('prog', 'fc', 'plan', 'sp', 'clbit_map', 'n_vars', 'ps', 'name', 'var_positions', 'pmf_map', 'pmf_order',
                 '_known_masses')


def _clone_sharded(payload, tables, fc):
    """Cached (plan, sharded plan) around fresh coefficient tables (plancache.PlanCache rebuild hook)."""
    import copy
    pl, sp = payload
    pl2 = copy.copy(pl)
    pl2.tables = tables[0]
    pl2.global_phase = fc.global_phase
    sp2 = copy.copy(sp)
    segs, k = [], 1
    for seg in sp.segments:
        if seg[0] == 'run':
            segs.append(('run', seg[1], tables[k], seg[3]))
            k += 1
        elif seg[0] == 'xblock':
            segs.append(('xblock', seg[1], seg[2], tables[k], seg[4]))
            k += 1
        else:
            segs.append(seg)
    sp2.segments = segs
    return pl2, sp2


class ShardedSimulator:
    """One rank of a statevector sharded on its g highest physical qubits over the
    2^g ranks of the default (or given) process group.  Same surface as B200Simulator for
    what bench.py and the tests use: prepare / execute / run / exact / close."""

    def __init__(self, precision='single', fusion='blocked', block_max=4, device=0, seed=None, group=None,
                 staging_bytes=1 << 30, name='qasm_simulator', layout='auto', expand_max=8, exchange='nccl',
                 plan_cache=True):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.group = group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.g = self.world.bit_length() - 1
        if 1 << self.g != self.world:
            raise ValueError('world size %d is not a power of two' % self.world)
        self.precision = precision
        self.fusion = fusion
        self.block_max = block_max
        self.expand_max = expand_max
        self.device = device
        self.seed = seed
        self.staging_bytes = int(staging_bytes)
        if layout not in ('auto', 'canonical'):
            raise ValueError("layout must be 'auto' or 'canonical'")
        self.layout = layout      # auto: shard on control-only qubits when the circuit has them (no communication)
        if exchange not in ('nccl', 'p2p', 'p2p-inplace'):
            raise ValueError("exchange must be 'nccl', 'p2p' or 'p2p-inplace'")
        # 'p2p': a qubit swap followed by sweeps on the swapped-in qubits runs as ONE kernel that reads the
        # peers' shards over NVLink (CUDA IPC mapped) and writes a second local buffer -- needs 2x the
        # shard in memory; anything it cannot serve falls back to the NCCL all-to-all + local passes.
        # 'p2p-inplace': the same kernel writing over the rank's own slabs, ordered against the peers' reads by
        # per-tile flags in peer-mapped memory (k_block_gather_inplace) -- no second buffer, any shard size
        self.exchange = exchange
        self._flags = None         # p2p-inplace: local flag tensor; _peer_flags: rank -> its address here
        self._peer_flags = None
        self._epoch = 0
        self._bufs = None          # p2p: [A, B] local state tensors
        self._peer_bufs = None     # p2p: rank -> [A, B] device addresses mapped from that rank (CUDA IPC)
        self._ipc_open = {}
        self._cur = 0
        self._name = name
        self._h = None
        self._state = None
        self._stage = None
        self._n_local = None
        self._profile = []
        self._launches_closed = 0
        self.exchange_ms = 0.0
        self.exchange_bytes = 0
        self.breakdown_ms = {}
        self.sync_before_exchange = False
        self._plan_cache = plancache.PlanCache() if plan_cache else None

    # ---- storage ---------------------------------------------------------------------------
    def _tensor_device(self):
        return self.torch.device('cuda', self.device)

    def _alloc_state(self, n_local):
        """(handle, flat real tensor of 2 * 2^n_local elements aliasing the state)."""
        t = self.torch
        rdt = t.float32 if self.precision in ('single', 'c64', 32) else t.float64
        state = t.empty(2 << n_local, dtype=rdt, device=self._tensor_device())
        h = _native.Handle(n_local, self.precision, self.device, ext_state_ptr=state.data_ptr())
        return h, state

    def _handle(self, n_local):
        if self._h is not None and self._n_local == n_local:
            return self._h
        self.close()
        self._h, self._state = self._alloc_state(n_local)
        self._n_local = n_local
        if self.exchange in ('p2p', 'p2p-inplace') and self._state.is_cuda:
            try:
                self._map_peers()
            except Exception as e:                       # IPC not available: stay on NCCL
                self._bufs = self._peer_bufs = None
                self.p2p_error = repr(e)
        return self._h

    def _map_peers(self):
        """Second local buffer + CUDA-IPC mappings of every rank's two buffers, opened with THIS rank's
        GPU current (qcm_ipc_open: cudaIpcOpenMemHandle + lazy peer access, the way NCCL's P2P transport
        maps its peers), so kernels launched here dereference them over NVLink."""
        t, dist = self.torch, self.dist
        inplace = self.exchange == 'p2p-inplace'
        if inplace:
            self._bufs = [self._state]
            words = max(_native.gather_flag_words(self._n_local, s, self.precision) for s in range(1, min(self.g, 3) + 1))
            self._flags = t.zeros(words, dtype=t.int32, device=self._state.device)
            self._flag_words = words
        else:
            self._bufs = [self._state, t.empty_like(self._state)]
        self._cur = 0
        meta = [_native.ipc_export(self.device, x.data_ptr()) for x in self._bufs + ([self._flags] if inplace else [])]
        gathered = [None] * self.world
        dist.all_gather_object(gathered, meta, group=self.group)
        peer_ptrs = {}
        self._ipc_open = {}                              # handle bytes -> base address in this process
        err = None
        try:
            for r in range(self.world):
                if r == self.rank:
                    peer_ptrs[r] = [x.data_ptr() for x in self._bufs + ([self._flags] if inplace else [])]
                    continue
                ptrs = []
                for hd, off in gathered[r]:
                    if hd not in self._ipc_open:
                        self._ipc_open[hd] = _native.ipc_open(self.device, hd)
                    ptrs.append(self._ipc_open[hd] + off)
                peer_ptrs[r] = ptrs
        except Exception as e:
            err = repr(e)
        errs = [None] * self.world
        dist.all_gather_object(errs, err, group=self.group)      # all ranks take the same path
        if any(errs):
            self._unmap_peers()
            raise RuntimeError('peer mapping failed: %s' % [e for e in errs if e][0])
        if inplace:
            self._peer_flags = {r: p[-1] for r, p in peer_ptrs.items()}
            peer_ptrs = {r: p[:-1] for r, p in peer_ptrs.items()}
        self._peer_bufs = peer_ptrs

    def _unmap_peers(self):
        if getattr(self, '_ipc_open', None):
            for base in self._ipc_open.values():
                try:
                    _native.ipc_close(self.device, base)
                except Exception:
                    pass
            self._ipc_open = {}
            try:
                self.torch.cuda.synchronize()
                self.dist.barrier(group=self.group)      # nobody frees a buffer a peer still has mapped
            except Exception:
                pass

    def close(self):
        if self._h is not None:
            try:
                self._launches_closed += self._h.timing()['kernel_launches']
            except Exception:
                pass
            self._h.close()
        self._unmap_peers()
        self._h = self._state = self._stage = None
        self._bufs = self._peer_bufs = self._flags = self._peer_flags = None
        self._n_local = None

    # ---- preparation -----------------------------------------------------------------------
    def prepare(self, circuit, n_vars=None):
        prog = ir.lower(circuit)
        fc = fusion.fuse(prog, 'off' if self.fusion == 'off' else 'clique')
        lazy = self.fusion == 'blocked'
        ng = 0
        if lazy and self.layout == 'auto' and len(fusion.control_only_qubits(fc)) >= self.g:
            ng = self.g
        fuse_x = self.exchange in ('p2p', 'p2p-inplace')

        def build(f):
            p, q = plan_for_shards(f, self.g, self.rank, lazy, self.block_max, ng, max(self.block_max, self.expand_max), fuse_x)
            tabs = [p.tables] + [seg[2] if seg[0] == 'run' else seg[3] for seg in q.segments if seg[0] in ('run', 'xblock')]
            return (p, q), tabs

        if self._plan_cache is None:
            pl, sp = build(fc)[0]
        else:
            # same structure as an earlier circuit (a theta / beta sweep): reuse plan + per-rank rewrite, refresh tables
            pl, sp = self._plan_cache.get(fc, ('sharded', lazy, self.block_max, self.expand_max, ng, self.g, self.rank, fuse_x),
                                          build, _clone_sharded)
        pr = _ShardPrepared()
        pr.prog, pr.fc, pr.plan, pr.sp, pr.name = prog, fc, pl, sp, prog.name

        def position(q):
            p = pl.layout[q]
            return sp.pos[p] if p < pl.n_phys else -1
        pr.clbit_map = np.full(prog.n_clbits, -1, dtype=np.int32)
        for c, q in prog.measures.items():
            pr.clbit_map[c] = position(q)
        if n_vars is None:
            n_vars = prog.metadata.get('num_vertices')
        pr.n_vars, pr.ps, pr.var_positions, pr.pmf_map, pr.pmf_order = n_vars, None, None, None, None
        if n_vars is not None:
            mask = 0
            for q in range(n_vars, prog.n_qubits):
                if position(q) >= 0:
                    mask |= 1 << position(q)
            pr.ps = (mask, 0, n_vars)
            pr.var_positions = [position(q) for q in range(n_vars)]
        return pr

    # ---- execution -------------------------------------------------------------------------
    def _exchange(self, betas):
        """Qubit-swap all-to-all: global qubits (rank bits ``betas``) <-> the top len(betas) local qubits."""
        t, dist = self.torch, self.dist
        s = len(betas)
        nl = self._n_local
        slab = 1 << (nl - s)
        st = self._state.view(1 << s, slab, 2)
        c_me = sum(((self.rank >> b) & 1) << i for i, b in enumerate(betas))
        base = self.rank
        for b in betas:
            base &= ~(1 << b)
        peers = []
        for j in range(1 << s):
            if j != c_me:
                pr = base
                for i, b in enumerate(betas):
                    pr |= ((j >> i) & 1) << b
                peers.append((j, pr))
        esz = self._state.element_size() * 2
        chunk = max(1, min(slab, self.staging_bytes // (2 * len(peers) * esz)))
        if chunk >= 1 << 16:
            chunk &= ~((1 << 16) - 1)       # keep every send/recv buffer 512 KiB-aligned (NCCL's fast path)
        if self._stage is None or self._stage.shape[1] < len(peers) or self._stage.shape[2] < chunk:
            self._stage = t.empty((2, len(peers), chunk, 2), dtype=self._state.dtype, device=self._state.device)
        stage = self._stage
        grank = (lambda r: r) if self.group is None else (lambda r: dist.get_global_rank(self.group, r))
        pending = None
        n_chunks = (slab + chunk - 1) // chunk
        for ci in range(n_chunks + 1):
            works = None
            if ci < n_chunks:
                off = ci * chunk
                n = min(chunk, slab - off)
                buf = stage[ci & 1]
                ops = []
                for k, (j, pr) in enumerate(peers):
                    ops.append(dist.P2POp(dist.isend, st[j, off:off + n], grank(pr), group=self.group))
                    ops.append(dist.P2POp(dist.irecv, buf[k, :n], grank(pr), group=self.group))
                works = (dist.batch_isend_irecv(ops), off, n, ci & 1)
            if pending is not None:
                ws, poff, pn, pb = pending
                for w in ws:
                    w.wait()
                for k, (j, pr) in enumerate(peers):
                    st[j, poff:poff + pn].copy_(stage[pb, k, :pn])
            pending = works
        self.exchange_bytes += len(peers) * slab * esz

    def _run_segments(self, sp, keep_flags=True):
        h = self._handle(sp.n_local)
        t = self.torch
        self._profile = []
        self.exchange_ms = 0.0
        self.exchange_bytes = 0
        for seg in sp.segments:
            if seg[0] == 'run':
                _, ops, tabs, mask = seg
                if not keep_flags and ops['flags'].any():
                    ops = ops.copy()
                    ops['flags'] &= ~fusion.QCM_FLAG_SAMPLE_CHECKPOINT     # no shots follow: skip the sampler's checkpoint tree
                h.set_shard(sp.g, sp.rank & mask)
                h.run_program(ops, tabs)
                if not getattr(h, 'deferred', False):       # reading an enqueued program's per-launch events would wait for it
                    self._profile.extend(h.op_profile())
            elif seg[0] == 'xblock' and self._peer_bufs is not None:
                _, betas, ops, tabs, mask = seg
                ms = self._gather_block(h, sp, betas, ops, tabs, mask)
                by = self._state.element_size() * (2 << sp.n_local)
                self._profile.append((-2, ms, by, by))
                self.exchange_ms += ms
            else:
                if self.sync_before_exchange:
                    self.dist.barrier(group=self.group)        # measurement aid: keep rank skew out of exchange_ms
                if self._state.is_cuda:
                    e0, e1 = t.cuda.Event(enable_timing=True), t.cuda.Event(enable_timing=True)
                    e0.record()
                    self._exchange(seg[1])
                    e1.record()
                    e1.synchronize()
                    ms = e0.elapsed_time(e1)
                else:
                    t0 = time.perf_counter()
                    self._exchange(seg[1])
                    ms = (time.perf_counter() - t0) * 1e3
                self.exchange_ms += ms
                sent = ((1 << len(seg[1])) - 1) * (1 << (sp.n_local - len(seg[1]))) * self._state.element_size() * 2
                self._profile.append((-1, ms, sent, sent))
                if seg[0] == 'xblock':                         # no peer mapping: all-to-all, then the sweeps locally
                    _, _, ops, tabs, mask = seg
                    h.set_shard(sp.g, sp.rank & mask)
                    h.run_program(ops, tabs)
                    self._profile.extend(h.op_profile())
        h.set_shard(sp.g, sp.rank & sp.mat_mask)
        return h

    def _gather_block(self, h, sp, betas, ops, tabs, mask):
        """Fused qubit swap + sweeps on the swapped-in qubits: one kernel reading the peers' current
        buffers (slab c_me of the rank with coordinate j, for every j) and writing this rank's other buffer."""
        t, dist = self.torch, self.dist
        s = len(betas)
        c_me = sum(((self.rank >> b) & 1) << i for i, b in enumerate(betas))
        base = self.rank
        for b in betas:
            base &= ~(1 << b)
        slab_bytes = self._state.element_size() * (2 << (sp.n_local - s))
        src, peers = [], []
        for j in range(1 << s):
            pr = base
            for i, b in enumerate(betas):
                pr |= ((j >> i) & 1) << b
            peers.append(pr)
            src.append(self._peer_bufs[pr][self._cur] + c_me * slab_bytes)
        t.cuda.synchronize()
        dist.barrier(group=self.group)          # every peer has finished writing the buffers read below
        e0, e1 = t.cuda.Event(enable_timing=True), t.cuda.Event(enable_timing=True)
        e0.record()
        h.set_shard(sp.g, sp.rank & mask)
        inplace = self._peer_flags is not None
        err = None
        try:
            if inplace:
                # in place: the kernels of all ranks order their overwrites behind each other's reads with flags
                self._epoch += 1
                h.run_gather_block_inplace(ops, tabs, src, [self._peer_flags[pr] for pr in peers], self._flag_words, self._epoch)
            else:
                dst = self._bufs[1 - self._cur]
                h.run_gather_block(ops, tabs, src, dst.data_ptr())
        except Exception as e:                  # noqa: BLE001 -- every rank must reach the barrier below, then fail together
            err = e
        e1.record()
        t.cuda.synchronize()
        # every peer's kernel is done: its signals and reads are behind us / it has finished reading this rank's old buffer
        bad = t.tensor([1 if err is not None else 0], dtype=t.int32, device=self._state.device)
        dist.all_reduce(bad, op=dist.ReduceOp.MAX, group=self.group)
        if int(bad.item()):
            raise RuntimeError('fused exchange failed on %s: %r' % ('this rank' if err is not None else 'a peer', err))
        if not inplace:
            self._cur = 1 - self._cur
            self._state = dst
        return e0.elapsed_time(e1)

    def _is_replica(self, sp):
        """This rank only mirrors another one (a global qubit that never materialised has bit 1 here)."""
        return (sp.rank & ~sp.mat_mask) != 0

    def _reduce(self, arr, op='sum'):
        t, dist = self.torch, self.dist
        dev = self._state.device
        x = t.from_numpy(np.ascontiguousarray(arr)).to(dev)
        dist.all_reduce(x, op=dist.ReduceOp.SUM, group=self.group)
        return x.cpu().numpy()

    def execute_deferred(self, pr, shots, seed=0, stream=0):
        """Run the gate program and ENQUEUE the result handling; returns a zero-argument callable that finishes it and
        returns what execute() returns.  Between the two the next circuit's program can be launched: a stream of
        circuits then pays the collective, the read-back and the host-side merge behind the next gate program instead
        of in front of it.  Falls back to plain execute() where the one-collective path does not apply."""
        sp = pr.sp
        replica = self._is_replica(sp)
        if not (pr.ps is not None and pr.n_vars <= 30 and shots and not replica):
            out = self.execute(pr, shots, seed, stream)
            return lambda: out
        t0 = time.perf_counter()
        known = self._known_rank_masses(pr)
        # no exchange in the plan and the one-collective path ahead: the gate program is only ENQUEUED too (the engine's
        # deferred mode), so the host runs ahead of the GPU and consecutive circuits execute back to back
        async_program = (known is not None and self._state is not None and self._state.is_cuda and self._h is not None
                         and self._n_local == sp.n_local and hasattr(self._h, 'tree_total_device')
                         and all(seg[0] == 'run' for seg in sp.segments) and self._device_path_ok(pr))
        if async_program:
            self._h.set_deferred(True)
        try:
            h = self._run_segments(sp, keep_flags=True)
            t1 = time.perf_counter()
            if not (self._state.is_cuda and hasattr(h, 'postselect_device') and self._device_path_ok(pr)):
                out = self._finish_general(h, pr, shots, seed, stream, replica, True, t0, t1)
                return lambda: out
            if known is None:
                out = self._finish_on_device(h, pr, shots, seed, stream, replica)
                return lambda: out
            rec = self._enqueue_one_collective(h, pr, shots, seed, stream, known)
        finally:
            if async_program:
                self._h.set_deferred(False)
        self.breakdown_ms = {'program': (t1 - t0) * 1e3, 'results enqueued (deferred)': (time.perf_counter() - t1) * 1e3}

        def finish():
            out = self._collect_one_collective(rec)
            if out is None:
                raise RuntimeError('a measured rank mass contradicts the plan; results of a deferred execution cannot be '
                                   'recomputed (the state has moved on): use execute()')
            return out
        return finish

    def execute(self, pr, shots, seed=0, stream=0, want_probs=True):
        """Returns (keys or None, probs or None, kept or None); identical on every rank."""
        sp = pr.sp
        t0 = time.perf_counter()
        h = self._run_segments(sp, keep_flags=bool(shots))
        t1 = time.perf_counter()
        replica = self._is_replica(sp)
        if (want_probs and pr.ps is not None and pr.n_vars <= 30 and shots and self._state.is_cuda
                and hasattr(h, 'postselect_device') and self._device_path_ok(pr)):
            keys, probs, kept = self._finish_on_device(h, pr, shots, seed, stream, replica)
            t2 = time.perf_counter()
            self.breakdown_ms = {'program': (t1 - t0) * 1e3, 'results (device path)': (t2 - t1) * 1e3}
            return keys, probs, kept
        return self._finish_general(h, pr, shots, seed, stream, replica, want_probs, t0, t1)

    def _finish_general(self, h, pr, shots, seed, stream, replica, want_probs, t0, t1):
        probs = kept = masses = None
        mass = None
        if shots:
            mass = 0.0 if replica else h.sample_prepare()
        if want_probs and pr.ps is not None and pr.n_vars <= 30:
            probs, kept, masses = self._postselect(h, pr, replica, mass)
        t2 = time.perf_counter()
        keys = None
        if shots:
            if masses is None:
                mvec = np.zeros(self.world)
                mvec[self.rank] = mass
                masses = self._reduce(mvec)
            # replicas mirror a rank that is sampling: they contribute nothing
            if replica:
                k = np.zeros(shots, dtype=np.int64)
            else:
                kk, mine = h.sample_sharded(shots, seed, stream, masses, pr.clbit_map if len(pr.clbit_map) else None)
                k = np.where(mine, kk, 0).astype(np.int64)
            keys = self._reduce(k).astype(np.uint64)
        self.breakdown_ms = {'program': (t1 - t0) * 1e3, 'postselect': (t2 - t1) * 1e3,
                             'sample': (time.perf_counter() - t2) * 1e3}
        return keys, probs, kept

    def _pmf_map(self, pr):
        """Where this rank's post-selected block lands in the 2^n pmf: (m, slice) when it is a
        contiguous run (local variables are qubits 0..m-1, global ones the higher variables in
        order -- the layouts the planner produces), else (m, index array)."""
        n, sp = pr.n_vars, pr.sp
        vp = pr.var_positions
        local_v = [q for q in range(n) if 0 <= vp[q] < sp.n_local]
        glob_v = [q for q in range(n) if vp[q] >= sp.n_local]
        m = len(local_v)
        if [vp[q] for q in local_v] != list(range(m)) or any(vp[q] < 0 for q in range(n)):
            raise NotImplementedError('post-selected vector needs the local variable qubits on positions 0..m-1')
        off = 0
        for q in glob_v:
            off |= ((sp.rank >> (vp[q] - sp.n_local)) & 1) << q
        if local_v == list(range(m)):
            return m, slice(off, off + (1 << m))
        loc = np.arange(1 << m, dtype=np.int64)
        idx = np.full(1 << m, off, dtype=np.int64)
        for j, q in enumerate(local_v):
            idx |= ((loc >> j) & 1) << q
        return m, idx

    def _device_path_ok(self, pr):
        """The ranks' pmf blocks tile the pmf (every global qubit a variable, no replicas): the layout
        the planner produces for QCMRF circuits -- results can then stay on the GPU until the end."""
        if pr.pmf_map is None:
            try:
                pr.pmf_map = self._pmf_map(pr)
            except NotImplementedError:
                pr.pmf_map = 'general'                      # variables anywhere: _postselect_general
        if pr.pmf_map == 'general':
            return False
        m, where = pr.pmf_map
        if pr.pmf_order is None:
            tiles = isinstance(where, slice) and where.stop - where.start == 1 << m and self._slices_tile(pr, m)
            pr.pmf_order = self._slice_order(pr, m) if tiles else False
        return bool(pr.pmf_order)

    def _known_rank_masses(self, pr):
        """Total probability mass of every rank when it follows from the plan alone: in the communication-free layout
        the global qubits are control-only product-state qubits (fusion.control_only_qubits), every later sweep is a
        unitary selected by them, so rank r holds exactly  prod_p |v_p[r_p]|^2  (times the norm of the local product
        state).  The sampler can then start without waiting for an all-gather of measured masses; the measured ones
        travel with the results and are checked against these.  None when the layout gives no such guarantee."""
        hit = getattr(pr, '_known_masses', False)
        if hit is not False:
            return hit
        pl, sp = pr.plan, pr.sp
        out = None
        if pl.n_global == self.g and self.g and len(pl.global_init) == self.g and len(pl.ops) and \
                int(pl.ops[0]['kind']) == fusion.QCM_OP_INIT_PRODUCT and sp.mat_mask == (1 << self.g) - 1:
            n_init = int(pl.ops[0]['n_active_out'])
            off = int(pl.ops[0]['table_off'])
            qv = pl.tables[off:off + 4 * max(n_init, 1)].reshape(-1, 4)
            norm = float(np.prod((qv[:n_init] ** 2).sum(axis=1))) if n_init else 1.0
            out = np.full(self.world, norm)
            for p, v in pl.global_init.items():
                w = np.abs(np.asarray(v, dtype=np.complex128)) ** 2
                for r in range(self.world):
                    out[r] *= w[(r >> (p - sp.n_local)) & 1]
            if not (out > 0).all():
                out = None
        pr._known_masses = out
        return out

    def _enqueue_one_collective(self, h, pr, shots, seed, stream, known):
        """Results of a sharded circuit with ONE collective: the rank masses are known from the plan
        (_known_rank_masses), so post-selection and sampling run back to back and a single all-gather carries every
        rank's pmf block, kept mass, measured mass and its shots' keys (0 where the shot landed elsewhere), followed
        by one read into pinned memory.  Everything is only ENQUEUED here; the returned record is finished by
        _collect_one_collective -- in between the next circuit's gate program can already run (the device buffers
        are reused in stream order, the pinned ones come from a ring of three)."""
        t, dist = self.torch, self.dist
        dev = self._state.device
        m, _ = pr.pmf_map
        nb = 1 << m
        words = nb + 3 + shots
        key = ('one', words)
        if getattr(self, '_dbuf_key', None) != key:
            self._dbuf = {
                'mine': t.zeros(words, dtype=t.float64, device=dev),
                'all': t.empty(self.world * words, dtype=t.float64, device=dev),
                'h_all': [t.empty(self.world * words, dtype=t.float64, pin_memory=True) for _ in range(3)],
                'h_small': [t.zeros(2, dtype=t.float64, pin_memory=True) for _ in range(3)],
                'flag': t.zeros(shots, dtype=t.uint8, device=dev),
                'slot': 0, 'busy': [None, None, None],
            }
            self._dbuf_key = key
        b = self._dbuf
        slot = b['slot']
        b['slot'] = (slot + 1) % 3
        old = b['busy'][slot]
        if old is not None and not old['done'].wait(timeout=60):
            # the pinned buffer of this slot still belongs to a deferred execution three circuits old
            raise RuntimeError('deferred executions must be finished (call what execute_deferred returned) before three '
                               'more are started')
        mask, value, _ = pr.ps
        base = b['mine'].data_ptr()
        h.postselect_device(mask, value, m, base, base + 8 * nb)
        h.tree_total_device(base + 8 * (nb + 1))             # this rank's measured mass, summed on the device
        h.sample_sharded_device(shots, seed, stream, known, pr.clbit_map if len(pr.clbit_map) else None,
                                base + 8 * (nb + 3), b['flag'].data_ptr())
        dist.all_gather_into_tensor(b['all'], b['mine'], group=self.group)
        b['h_all'][slot].copy_(b['all'], non_blocking=True)
        ev = t.cuda.Event()
        ev.record()
        import threading
        # the record keeps its buffers: a later circuit of another size replaces self._dbuf before this one is collected
        rec = {'event': ev, 'slot': slot, 'nb': nb, 'words': words, 'order': pr.pmf_order, 'done': threading.Event(),
               'known': known, 'bufs': b}
        b['busy'][slot] = rec
        return rec

    def _collect_one_collective(self, rec):
        """(keys, probs, kept) of an enqueued record, or None (consistently on every rank) if a measured rank mass
        contradicted the plan -- the caller then takes the general path."""
        b = rec['bufs']
        rec['event'].synchronize()
        nb, words = rec['nb'], rec['words']
        hall = b['h_all'][rec['slot']].numpy().reshape(self.world, words)
        # the measured rank masses (gathered with the results: every rank sees all of them) against the plan's
        tol = 1e-9 if self.precision in ('double', 'c128', 64) else 2e-5
        ok = bool((np.abs(hall[:, nb + 1] - rec['known']) <= tol * rec['known']).all())
        out = None
        if ok:
            kept = float(hall[:, nb].sum())
            blocks = hall[:, :nb]
            if rec['order'] != list(range(self.world)):
                blocks = blocks[rec['order']]
            probs = np.array(blocks, order='C').reshape(-1)          # always a copy: the pinned buffer is reused
            keys = hall[:, nb + 3:].view(np.int64).sum(axis=0).astype(np.uint64)
            out = (keys, probs, kept)
        rec['done'].set()                                    # the pinned buffer of this slot may be reused
        return out

    def _finish_one_collective(self, h, pr, shots, seed, stream, known):
        return self._collect_one_collective(self._enqueue_one_collective(h, pr, shots, seed, stream, known))

    def _finish_on_device(self, h, pr, shots, seed, stream, replica):
        """Post-selection, all-gather of (pmf block, kept, mass), sharded sampling and the key merge with
        every intermediate on the GPU (the sampler reads the gathered rank masses in place): one final read of
        pmf + keys into pinned memory is the only synchronisation."""
        t, dist = self.torch, self.dist
        dev = self._state.device
        known = None if replica else self._known_rank_masses(pr)
        if known is not None:
            out = self._finish_one_collective(h, pr, shots, seed, stream, known)
            if out is not None:
                return out
        m, _ = pr.pmf_map
        blk = (1 << m) + 2
        key = (blk, shots)
        if getattr(self, '_dbuf_key', None) != key:
            self._dbuf = {
                'mine': t.zeros(blk, dtype=t.float64, device=dev),
                'all': t.empty(self.world * blk, dtype=t.float64, device=dev),
                'keys': t.zeros(shots, dtype=t.int64, device=dev),
                'flag': t.zeros(shots, dtype=t.uint8, device=dev),
                'h_all': t.empty(self.world * blk, dtype=t.float64, pin_memory=True),
                'h_keys': t.empty(shots, dtype=t.int64, pin_memory=True),
            }
            self._dbuf_key = key
        b = self._dbuf
        mask, value, _ = pr.ps
        if replica:
            b['mine'].zero_()
        else:
            mass = h.sample_prepare()
            h.postselect_device(mask, value, m, b['mine'].data_ptr(), b['mine'].data_ptr() + 8 * (1 << m))
            b['mine'][-1:].fill_(mass)
        dist.all_gather_into_tensor(b['all'], b['mine'], group=self.group)
        b['h_all'].copy_(b['all'], non_blocking=True)
        if replica:
            b['keys'].zero_()
        elif hasattr(h, 'sample_sharded_devmass'):
            # the sampler reads the gathered rank masses where the all-gather left them: nothing comes back to the
            # host between the two collectives (keys of shots that landed on another rank are written as 0)
            h.sample_sharded_devmass(shots, seed, stream, b['all'].data_ptr() + 8 * (blk - 1), blk, self.world,
                                     pr.clbit_map if len(pr.clbit_map) else None, b['keys'].data_ptr(), b['flag'].data_ptr())
        else:
            masses = b['all'].view(self.world, blk)[:, -1].cpu().numpy()
            h.sample_sharded_device(shots, seed, stream, masses, pr.clbit_map if len(pr.clbit_map) else None,
                                    b['keys'].data_ptr(), b['flag'].data_ptr())
        dist.all_reduce(b['keys'], op=dist.ReduceOp.SUM, group=self.group)
        b['h_keys'].copy_(b['keys'], non_blocking=True)
        t.cuda.current_stream(dev).synchronize()
        hall = b['h_all'].numpy().reshape(self.world, blk)
        kept = float(hall[:, -2].sum())
        blocks = hall[:, :-2]
        if pr.pmf_order != list(range(self.world)):
            blocks = blocks[pr.pmf_order]
        probs = np.array(blocks, order='C').reshape(-1)          # always a copy: the pinned buffer is reused
        keys = b['h_keys'].numpy().astype(np.uint64)
        return keys, probs, kept

    def _postselect(self, h, pr, replica, mass=None):
        """Exact post-selected pmf (index: variable q <-> bit q) and success probability, on every rank.
        Variables on local positions 0..m-1 come from the engine's contiguous reduction; variables on
        global positions select which part of the pmf this rank owns.  One all-gather moves every
        rank's block, its kept mass and (for the sampler) its total mass.  Returns (pmf, kept, masses)."""
        n = pr.n_vars
        if pr.pmf_map is None:
            try:
                pr.pmf_map = self._pmf_map(pr)
            except NotImplementedError:
                pr.pmf_map = 'general'
        if pr.pmf_map == 'general':
            return self._postselect_general(h, pr, replica, mass)
        m, where = pr.pmf_map
        mask, value, _ = pr.ps
        mine = np.zeros((1 << m) + 2)
        if not replica:
            p, k = h.postselect(mask, value, m)
            mine[:-2] = p
            mine[-2] = k
            mine[-1] = 0.0 if mass is None else mass
        t, dist = self.torch, self.dist
        x = t.from_numpy(mine).to(self._state.device)
        allx = t.empty(self.world * mine.size, dtype=x.dtype, device=x.device)
        dist.all_gather_into_tensor(allx, x, group=self.group)
        allx = allx.cpu().numpy().reshape(self.world, mine.size)
        masses = allx[:, -1].copy()
        kept = float(allx[:, -2].sum())
        if pr.pmf_order is None:
            tiles = isinstance(where, slice) and where.stop - where.start == 1 << m and self._slices_tile(pr, m)
            pr.pmf_order = self._slice_order(pr, m) if tiles else False
        if pr.pmf_order:
            # rank r's block is pmf[r_off : r_off + 2^m]; the blocks tile the pmf
            blocks = allx[:, :-2]
            if pr.pmf_order != list(range(self.world)):
                blocks = blocks[pr.pmf_order]
            return np.ascontiguousarray(blocks).reshape(-1), kept, masses
        out = np.zeros(1 << n)
        for r in range(self.world):
            wr = self._pmf_where_for_rank(pr, r, m)
            if wr is None:
                continue
            if isinstance(wr, slice):
                out[wr] += allx[r, :-2]
            else:
                np.add.at(out, wr, allx[r, :-2])
        return out, kept, masses

    def _postselect_general(self, h, pr, replica, mass=None):
        """The same result for ANY layout of the variable qubits (a foreign circuit whose first-use layout scatters
        them): every rank takes its whole masked local distribution from the engine, adds it into the 2^n pmf by index
        arithmetic on the host, and one all-reduce sums pmf, kept mass and the ranks' masses.  Small states only."""
        n, sp = pr.n_vars, pr.sp
        nl = sp.n_local
        if nl > 26 or n > 26:
            raise NotImplementedError('post-selected vector of a sharded state this large needs the variable qubits on the '
                                      'low local positions')
        mask, value, _ = pr.ps
        mine = np.zeros((1 << n) + self.world + 1)
        if not replica:
            full, k = h.postselect(mask, value, nl)
            idx = np.arange(1 << nl, dtype=np.int64)
            oi = np.zeros(1 << nl, dtype=np.int64)
            for q in range(n):
                p = pr.var_positions[q]
                if p < 0:
                    continue                                # never materialised: the variable reads 0
                if p < nl:
                    oi |= ((idx >> p) & 1) << q
                else:
                    oi |= ((sp.rank >> (p - nl)) & 1) << q
            np.add.at(mine[:1 << n], oi, full)
            mine[(1 << n) + self.rank] = 0.0 if mass is None else mass
            mine[-1] = k
        tot = self._reduce(mine)
        return tot[:1 << n].copy(), float(tot[-1]), tot[1 << n:-1].copy()

    def _pmf_where_for_rank(self, pr, r, m):
        """Index set of rank r's block in the pmf, or None if r is a replica."""
        sp = pr.sp
        if r & ~sp.mat_mask:
            return None
        n, vp = pr.n_vars, pr.var_positions
        local_v = [q for q in range(n) if 0 <= vp[q] < sp.n_local]
        off = 0
        for q in range(n):
            if vp[q] >= sp.n_local:
                off |= ((r >> (vp[q] - sp.n_local)) & 1) << q
        if local_v == list(range(m)):
            return slice(off, off + (1 << m))
        loc = np.arange(1 << m, dtype=np.int64)
        idx = np.full(1 << m, off, dtype=np.int64)
        for j, q in enumerate(local_v):
            idx |= ((loc >> j) & 1) << q
        return idx

    def _slices_tile(self, pr, m):
        """Do the ranks' blocks tile the pmf exactly once (every global qubit a variable, no replicas)?"""
        sp = pr.sp
        if sp.mat_mask != (1 << sp.g) - 1:
            return False
        offs = set()
        for r in range(self.world):
            w = self._pmf_where_for_rank(pr, r, m)
            if not isinstance(w, slice):
                return False
            offs.add(w.start)
        return len(offs) == self.world and (self.world << m) == (1 << pr.n_vars)

    def _slice_order(self, pr, m):
        return sorted(range(self.world), key=lambda r: self._pmf_where_for_rank(pr, r, m).start)

    def run(self, circuits, shots=1024, seed=None, n_vars=None):
        from .backend import Job, Result, _keys_to_counts, _normalised
        t0 = time.perf_counter()
        single = not isinstance(circuits, (list, tuple))
        circs = [circuits] if single else list(circuits)
        if seed is None:
            seed = self.seed if self.seed is not None else 0
        def entry(c, pr, i, finish, exchange_ms):
            keys, probs, kept = finish()
            counts = _keys_to_counts(keys, pr.prog.n_clbits) if shots else None
            h2d = sum(seg[1].nbytes + seg[2].nbytes for seg in pr.sp.segments if seg[0] == 'run')
            d2h = (probs.nbytes + 8 if probs is not None else 0) + (keys.nbytes if keys is not None else 0)
            pmf = _normalised(probs, kept)                 # in place, behind the next circuit's gate program
            return {'circuit': c, 'name': pr.name, 'counts': counts, 'probs': None if pmf is not None else probs, 'pmf': pmf, 'kept': kept,
                    'meta': {'path': 'sharded', 'ranks': self.world, 'n_qubits': pr.prog.n_qubits,
                             'n_phys': pr.plan.n_phys, 'n_local': pr.sp.n_local, 'passes': pr.plan.n_passes,
                             'exchanges': pr.sp.n_exchanges, 'exchange_ms': exchange_ms,
                             'exchange_path': ('p2p-fused-inplace' if self._peer_flags is not None else 'p2p-fused')
                             if self._peer_bufs is not None else 'nccl',
                             'h2d_bytes': int(h2d), 'd2h_bytes': int(d2h), 'philox_stream': i}}

        entries = []
        if len(circs) > 1 and shots and self._state_is_cuda():
            # a list of circuits is a pipeline: circuit i+1 is prepared and its gate program enqueued BEFORE circuit i's
            # results are collected (collective + read-back awaited, keys merged, counts dict built), so the GPU works on
            # i+1 while the host finishes i.  One thread: eight ranks with a helper thread each oversubscribed the host.
            pend = None
            for i, c in enumerate(circs):
                pr = self.prepare(c, n_vars=n_vars)
                fin = self.execute_deferred(pr, int(shots), seed, i)
                if pend is not None:
                    entries.append(entry(*pend))
                pend = (c, pr, i, fin, self.exchange_ms)
            entries.append(entry(*pend))
        else:
            for i, c in enumerate(circs):
                pr = self.prepare(c, n_vars=n_vars)
                out = self.execute(pr, int(shots), seed, i)
                entries.append(entry(c, pr, i, lambda out=out: out, self.exchange_ms))
        return Job(Result(entries, single, self._name, seed, int(shots), time.perf_counter() - t0))

    def _state_is_cuda(self):
        return self._state is None or bool(getattr(self._state, 'is_cuda', False))

    def exact(self, circuit, n=None):
        return self.run(circuit, shots=0, n_vars=n).result().postselected_probabilities(0)

    # ---- introspection ---------------------------------------------------------------------
    def op_profile(self):
        return list(self._profile)

    def op_kernels(self):
        """Kernel names of the LAST run segment's ops (the segment that holds the dominant final pass)."""
        try:
            return self._h.op_kernels() if self._h is not None else []
        except Exception:
            return []

    def kernel_launches(self):
        live = self._h.timing()['kernel_launches'] if self._h is not None else 0
        return self._launches_closed + live

    def last_timing(self):
        return self._h.timing() if self._h is not None else None

    def local_amplitudes(self):
        return self._h.get_amplitudes()
