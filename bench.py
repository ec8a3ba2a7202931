#!/usr/bin/env python
"""Headline benchmark: QCMRF circuits/sec on the 34-qubit complex64 synthetic tree MRF
(BASELINE.json config 4; config 3's 33-qubit graph with --workload q33), with the
achieved HBM GB/s of the dominant gate pass against the measured B200 roofline and the
CPU restatement of the reference path timed beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

A step = one circuit: product-state init (+H layer), the fused clique passes, the
ancilla post-selection reduction with the exact 2^n pmf, and 10000 sampled shots
(the reference's SHOTS, run_experiment.py:16).  `value` times that with the fused
program already planned and its coefficient tables on the host (the state never
leaves HBM: it is 64 GiB, far beyond the 126 MB L2, so no L2 flush is needed); `e2e`
times the public call -- ``B200Simulator.run(QCMRF(cliques, theta), shots)`` from host
objects to a counts dict and the pmf in host memory, including lowering, fusion,
planning, table upload and result download -- with a fresh theta every step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

SHOTS = 10000
METRIC = 'QCMRF circuits/sec'


NCU_TRAFFIC_FILES = ('r02_ncu_prof_low.csv', 'r01_ncu_prof_low.csv')      # newest first


def ncu_traffic(workload, world):
    """(dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel, file) from the committed `ncu --set full`
    capture of this same workload (profiles/), or (None, None)."""
    if workload != 'q34' or world != 1:
        return None, None
    import csv
    for fn in NCU_TRAFFIC_FILES:
        try:
            tot = 0.0
            for row in csv.reader(open(os.path.join(ROOT, 'profiles', fn))):
                if row and row[0] in ('dram__bytes_read.sum', 'dram__bytes_write.sum'):
                    tot += float(row[2].replace(',', '')) * {'Gbyte': 1e9, 'Mbyte': 1e6, 'Kbyte': 1e3, 'byte': 1.0}[row[1]]
            if tot:
                return tot, 'profiles/' + fn
        except Exception:
            continue
    return None, None


def load_peaks():
    try:
        p = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        return float(p['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler:
    """SM clock, power and throttle reasons of one GPU DURING the timed region: NVML polled in-process every few
    milliseconds (a multi-GPU step is ~1.5 ms and `nvidia-smi -lms` needs a second to print its first line); the
    nvidia-smi subprocess is the fallback when the NVML binding is missing."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index=0, period_s=0.004):
        self.index = index
        self.period = period_s
        self.rows = []                       # (sm MHz, max MHz, watts, reasons bitmask or None)
        self.proc = None
        self.nv = None
        self.stop_flag = threading.Event()
        self.how = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates every GPU of the box; CUDA_VISIBLE_DEVICES may have renumbered them
            vis = os.environ.get('CUDA_VISIBLE_DEVICES')
            idx = self.index
            handle = None
            if vis:
                ids = [v.strip() for v in vis.split(',') if v.strip()]
                if idx < len(ids) and ids[idx].isdigit():
                    idx = int(ids[idx])
                elif idx < len(ids):
                    handle = pynvml.nvmlDeviceGetHandleByUUID(ids[idx].encode() if hasattr(pynvml, 'c_char_p') else ids[idx])
            self.nv = (pynvml, handle if handle is not None else pynvml.nvmlDeviceGetHandleByIndex(idx))
            self.how = 'nvml'
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        except Exception:
            self.nv = None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.how = 'nvidia-smi -lms 100'
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _poll(self):
        nv, h = self.nv
        try:
            smax = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        except Exception:
            smax = None
        reasons_fn = getattr(nv, 'nvmlDeviceGetCurrentClocksEventReasons', None) or getattr(nv, 'nvmlDeviceGetCurrentClocksThrottleReasons', None)
        while not self.stop_flag.is_set():
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    w = nv.nvmlDeviceGetPowerUsage(h) / 1e3
                except Exception:
                    w = None
                try:
                    rs = int(reasons_fn(h)) if reasons_fn else None
                except Exception:
                    rs = None
                self.rows.append((sm, smax, w, rs))
            except Exception:
                pass
            self.stop_flag.wait(self.period)

    def _read(self):
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        bits = {'hw_slowdown': 0x8, 'hw_thermal_slowdown': 0x40, 'sw_thermal_slowdown': 0x20, 'sw_power_cap': 0x4}
        for line in self.proc.stdout:
            r = [x.strip() for x in line.split(',')]
            if len(r) < 9:
                continue
            try:
                mask = 0
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith('active'):
                        mask |= bits[nm]
                self.rows.append((float(r[1]), float(r[2]), float(r[3]), mask))
            except ValueError:
                continue

    def mark(self):
        """Index of the next sample: bench.py brackets its timed regions with it."""
        return len(self.rows)

    def stop(self, lo=0, hi=None):
        """Summary over samples [lo, hi) -- the timed regions -- falling back to every sample when that window is empty."""
        self.stop_flag.set()
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        if self.how is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no NVML binding and no nvidia-smi']}
        if self.nv:
            self.th.join(timeout=1)
        rows = self.rows[lo:hi] or self.rows
        window = 'timed regions' if self.rows[lo:hi] else 'whole run (no sample fell inside the timed regions)'
        # NVML clocks-event-reason bits (nvml.h): sw_power_cap 0x4, hw_slowdown 0x8, sw_thermal 0x20, hw_thermal 0x40
        bits = {'sw_power_cap': 0x4, 'hw_slowdown': 0x8, 'sw_thermal_slowdown': 0x20, 'hw_thermal_slowdown': 0x40}
        reasons = sorted(nm for nm, b in bits.items() if any(r[3] is not None and (r[3] & b) for r in rows))
        sm = [r[0] for r in rows]
        smax = [r[1] for r in rows if r[1] is not None]
        power = [r[2] for r in rows if r[2] is not None]
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(smax) if smax else None,
                'power_w_max': max(power) if power else None, 'samples': len(sm), 'reasons': reasons,
                'how': self.how, 'window': window}


# ------------------------------------------------------------------------------------------
def _cpu_threads():
    cores = len(os.sched_getaffinity(0))
    # every host thread, also under torchrun (which exports OMP_NUM_THREADS=1 to its workers)
    os.environ['OMP_NUM_THREADS'] = str(cores)
    try:
        import ctypes
        ctypes.CDLL('libgomp.so.1').omp_set_num_threads(cores)
    except OSError:
        pass
    return cores


def _cpu_one(nv, seed, fused):
    """One circuit of the random-tree family with nv variables (N = 2 nv qubits) on the host cores, complex128:
    B1 (fused=False) = one OpenMP sweep of the dense state per gate of QCMRF._build's program (H, X, flagged MCX,
    CP -- QCMRF.py:204-243), what an UNFUSED statevector simulator does for run_experiment.py:56; B2 (fused=True)
    = the GPU path's fused program at full width (H layer + one multiplexer sweep per clique).  Both include the
    post-selection reduction and 10000 shots.  Returns (seconds, N, sweeps)."""
    from oracle import cbridge, program
    from qcmrf_b200 import workloads
    Cs = workloads.random_tree(nv, 0)
    th = workloads.theta_for(Cs)
    n_s, k_s, N_s, _ = program.sizes(Cs)
    tabs = None
    if fused:
        arr, n_ops, tabs, _N = cbridge.compile_fused(Cs, theta=th)
    else:
        ops_s, _ = program.qcmrf_program(Cs, th)
        arr, n_ops, _meas = cbridge.compile_unfused(ops_s)
    mask = ((1 << N_s) - 1) & ~((1 << n_s) - 1)
    t0 = time.perf_counter()
    psi = cbridge.run(N_s, arr, n_ops, tabs)
    cbridge.postselect(N_s, psi, mask, 0, n_s)
    cbridge.sample(N_s, psi, SHOTS, seed)
    dt = time.perf_counter() - t0
    del psi
    return dt, N_s, n_ops


def _fit_per_sweep(ladder):
    """log2(seconds per sweep) = a + b N, least squares over the ladder; returns (a, b, worst |residual| in log2)."""
    N = np.array([r['N'] for r in ladder], dtype=np.float64)
    y = np.log2(np.array([r['s'] / r['sweeps'] for r in ladder]))
    if len(N) < 2:
        return float(y[0] - N[0]), 1.0, 0.0
    b, a = np.polyfit(N, y, 1)
    return float(a), float(b), float(np.abs(a + b * N - y).max())


def cpu_reference(target_cliques, steps=1, warmup=0, budget_s=75.0, ram_bytes=None):
    """The reference path on the host cores, MEASURED on a ladder of the same family (random tree MRFs at
    N = 24, 26, 28, 30 total qubits, complex128, every host thread): B1 unfused (Aer without gate fusion: an
    upper bound on Aer's time, which fuses up to 5-qubit blocks), B2 fused (the GPU path's program on the CPU:
    a lower bound).  The 34-qubit target (256 GiB complex128) cannot be held on the host: its time is
    EXTRAPOLATED from the fitted slope of log2(seconds per sweep) against N, with the fit's residual printed,
    and flagged `extrapolated`.  A rung is skipped when the fit so far predicts it would blow the time budget
    or when the state would not fit in half the host RAM."""
    from oracle import program
    from qcmrf_b200 import workloads
    cores = _cpu_threads()
    if ram_bytes is None:
        try:
            ram_bytes = os.sysconf('SC_PHYS_PAGES') * os.sysconf('SC_PAGE_SIZE')
        except (ValueError, OSError):
            ram_bytes = 32 << 30
    n_t, k_t, N_t, _ = program.sizes(target_cliques)
    ops_t, _ = program.qcmrf_program(target_cliques, workloads.theta_for(target_cliques))
    g_b1 = sum(1 for g in ops_t if g[0] not in ('measure', 'barrier'))
    g_b2 = n_t + k_t
    t_start = time.perf_counter()
    ladders = {'b1': [], 'b2': []}
    for fused, key, share in ((True, 'b2', 0.2), (False, 'b1', 1.0)):
        for nv in (12, 13, 14, 15):
            N_s = 2 * nv
            if (16 << N_s) > ram_bytes // 2:
                break
            lad = ladders[key]
            if lad:
                a, b, _r = _fit_per_sweep(lad) if len(lad) > 1 else (np.log2(lad[0]['s'] / lad[0]['sweeps']) - lad[0]['N'], 1.0, 0)
                predicted = 2.0 ** (a + b * N_s) * lad[-1]['sweeps'] * 1.1
                if (time.perf_counter() - t_start) + predicted > budget_s * share + (0 if fused else budget_s * 0.2):
                    break
            dt, N_s, n_ops = _cpu_one(nv, 1984, fused)
            lad.append({'N': N_s, 'sweeps': n_ops, 's': dt})
    # the reference arm's timed steps: repeat the largest unfused rung that keeps the whole run short
    b1 = ladders['b1']
    rep = b1[-1]
    for r in b1:
        if r['s'] * (steps + warmup) <= 60.0:
            rep = r
    times = []
    for it in range(warmup + steps - 1):              # the ladder run of this rung counts as the first step
        dt, _N, _ops = _cpu_one(rep['N'] // 2, 1984 + it, False)
        if it >= warmup - 1:
            times.append(dt)
    times.append(rep['s'])
    rep_s = float(np.mean(times))
    out = {}
    for key, g_t in (('b1', g_b1), ('b2', g_b2)):
        a, b, resid = _fit_per_sweep(ladders[key])
        t_target = 2.0 ** (a + b * N_t) * g_t
        out[key] = {'t_target': t_target, 'fit': {'log2_s_per_sweep_intercept': a, 'slope_per_qubit': b,
                                                  'worst_residual_log2': resid, 'target_sweeps': g_t}}
    # the timed rung, scaled by the fitted slope (not the ideal x2 per qubit) -- agrees with the fit at that rung
    t_target = out['b1']['t_target'] * (rep_s / rep['s'])
    sample = ('B1 = unfused port of the reference program, complex128, %d host threads; ladder of random-tree MRFs '
              'N=%s timed here (%s s/circuit); timed steps at N=%d (%d sweeps): %.3f s/circuit; the %d-qubit target '
              '(%d sweeps, 256 GiB complex128) is EXTRAPOLATED with the fitted slope 2^(%.3f N) per sweep (worst '
              'residual %.3f in log2)'
              % (cores, '/'.join(str(r['N']) for r in b1), '/'.join('%.2f' % r['s'] for r in b1), rep['N'], rep['sweeps'],
                 rep_s, N_t, g_b1, out['b1']['fit']['slope_per_qubit'], out['b1']['fit']['worst_residual_log2']))
    base = {'value': 1.0 / t_target, 'unit': 'circuits/s', 'cores': cores, 'kind': 'port', 'sample': sample,
            'extrapolated': True, 'variant': 'B1 unfused (one sweep per gate of QCMRF._build; Aer fuses gates, so this is an '
                                             'upper bound on Aer\'s time; B2 below is the lower bound)',
            'ladder': [dict(r, variant='b1') for r in b1] + [dict(r, variant='b2') for r in ladders['b2']],
            'fit_b1': out['b1']['fit'], 'fit_b2': out['b2']['fit'],
            'b2_value': 1.0 / out['b2']['t_target'], 'b2_seconds_per_circuit_extrapolated': out['b2']['t_target'],
            'seconds_per_circuit_extrapolated': t_target,
            'measured_not_extrapolated': {'N': rep['N'], 'seconds_per_circuit_b1': rep_s, 'circuits_per_s_b1': 1.0 / rep_s,
                                          'b2_seconds_per_circuit': next((r['s'] for r in ladders['b2'] if r['N'] == rep['N']), None)},
            'sample_seconds_per_circuit': rep_s, 'sample_amp_updates_per_sec': rep['sweeps'] * 2.0 ** rep['N'] / rep_s,
            'steps_timed': len(times), 'host_ram_gib': ram_bytes / 2.0 ** 30}
    return base, t_target


def run_reference_arm(args, cliques, N):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    base, t_target = cpu_reference(cliques, steps=max(1, args.steps), warmup=min(args.warmup, 1))
    line = {'impl': 'reference', 'metric': METRIC, 'value': base['value'], 'unit': 'circuits/s',
            'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': t_target * 1e3,
            'ms_per_step_kind': 'EXTRAPOLATED to the %d-qubit workload from the measured ladder (cpu_baseline.ladder, fit_b1); '
                                'the timed steps ran the N=%d member of the family: %.1f ms each'
                                % (N, base['measured_not_extrapolated']['N'], base['sample_seconds_per_circuit'] * 1e3),
            'extrapolated': True,
            'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': workload_config(args, cliques, N), 'cpu_baseline': base,
            'e2e': {'value': base['value'], 'unit': 'circuits/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line), flush=True)


def brute_force_pmf(cliques, theta, beta=1.0):
    """p(x) ~ exp(beta * sum_C theta[C, x_C]) by enumeration, index x_0 = MSB (eval.py:100-101), and
    delta = Z / 2^n -- the check printed with every bench line (plain numpy, independent of oracle/)."""
    n = max(max(c) for c in cliques) + 1
    x = np.arange(1 << n, dtype=np.int64)
    e = np.zeros(1 << n)
    off = 0
    for c in cliques:
        idx = np.zeros(1 << n, dtype=np.int64)
        for v in c:
            idx = (idx << 1) | ((x >> (n - 1 - v)) & 1)
        e += np.asarray(theta[off:off + (1 << len(c))], dtype=np.float64)[idx]
        off += 1 << len(c)
    w = np.exp(beta * e)
    return w / w.sum(), float(w.sum() / (1 << n))


def weissman_tv_bound(K, S, alpha):
    """P(TV > bound) <= alpha for S draws over K outcomes (SURVEY.md T5)."""
    return 0.5 * float(np.sqrt(2.0 * (K * np.log(2.0) + np.log(1.0 / alpha)) / S))


def shot_marginal_tv(cliques, theta, counts, beta=1.0):
    """Sampled histogram vs the exact distribution, through marginals that 10^4 shots can resolve: for every
    clique C the joint of (x_C, its ancilla) -- 2^(|C|+1) outcomes, exact law P(x_C = y, a = 0) =
    2^-|C| exp(beta theta_{C,y}), P(x_C = y, a = 1) = 2^-|C| (1 - exp(beta theta_{C,y})) (SURVEY App. A: x is
    uniform before post-selection).  Key layout of App. B (QCMRF.py:219,231,238-243): variable v = bit n-1-v,
    ancilla of clique ii = bit n+1+ii, bit n always 0.  Returns the worst TV, its Weissman bound at a union
    alpha of 1e-6 over the cliques, and whether bit n was ever set."""
    n = max(max(c) for c in cliques) + 1
    keys = np.fromiter((int(k, 2) for k in counts), dtype=np.uint64, count=len(counts))
    cnt = np.fromiter(counts.values(), dtype=np.float64, count=len(counts))
    S = cnt.sum()
    worst, off = 0.0, 0
    kmax = 2
    for ii, c in enumerate(cliques):
        m = len(c)
        y = np.zeros(len(keys), dtype=np.int64)
        for v in c:
            y = (y << 1) | ((keys >> np.uint64(n - 1 - v)) & np.uint64(1)).astype(np.int64)
        a = ((keys >> np.uint64(n + 1 + ii)) & np.uint64(1)).astype(np.int64)
        obs = np.bincount(y + (a << m), weights=cnt, minlength=2 << m) / S
        w = np.exp(beta * np.asarray(theta[off:off + (1 << m)], dtype=np.float64))
        exact = np.concatenate([w, 1.0 - w]) / (1 << m)
        worst = max(worst, 0.5 * float(np.abs(obs - exact).sum()))
        kmax = max(kmax, 2 << m)
        off += 1 << m
    scratch_set = bool(((keys >> np.uint64(n)) & np.uint64(1)).any())
    return worst, weissman_tv_bound(kmax, S, 1e-6 / len(cliques)), scratch_set


def parity_check(cliques, theta, p, delta, counts, beta=1.0, tol=1e-5, rel_tol=2e-4):
    """Last e2e step vs brute-force enumeration (plain numpy, independent of oracle/): the post-selected pmf --
    max |p - p_exact| (north-star absolute tolerance) AND max |p - p_exact| / p_exact (the absolute bound is
    vacuous at p ~ 2^-17), delta, and the sampled shots through the per-clique marginal TV and the kept fraction."""
    n = max(max(c) for c in cliques) + 1
    if n > 24:
        return {}
    pb, db = brute_force_pmf(cliques, theta, beta)
    out = {'max_abs_p_error_vs_brute_force': float(np.abs(p - pb).max()), 'rel_p_err': float((np.abs(p - pb) / pb).max()),
           'delta_error_vs_brute_force': abs(float(delta) - db), 'delta_rel_err': abs(float(delta) - db) / db,
           'tolerance': tol, 'rel_tolerance': rel_tol, 'exact_delta': db, 'argmax_ok': bool(np.argmax(p) == np.argmax(pb))}
    ok = out['max_abs_p_error_vs_brute_force'] < tol and out['rel_p_err'] < rel_tol and out['delta_rel_err'] < rel_tol
    if counts:
        S = sum(counts.values())
        kept = sum(v for k, v in counts.items() if int(k, 2) < (1 << n))
        tv, bound, scratch = shot_marginal_tv(cliques, theta, counts, beta)
        sd = float(np.sqrt(db * (1 - db) / S))
        out.update({'sampled_success_fraction': kept / max(S, 1), 'success_fraction_5sigma': 5 * sd + 1.0 / S,
                    'tv': tv, 'tv_bound': bound, 'tv_what': 'worst per-clique (x_C, ancilla) marginal of the sampled keys vs exact',
                    'scratch_clbit_ever_set': scratch})
        ok = ok and tv < bound and not scratch and abs(kept / S - db) < 5 * sd + 1.0 / S
    out['parity_ok'] = bool(ok)
    return out


def ranks_identical(dist, world, counts, p, delta):
    """Every rank must hold the same counts, pmf and delta (what tests/multi_gpu_worker.py asserts)."""
    import hashlib
    hsh = hashlib.sha256()
    if counts:
        hsh.update(json.dumps(sorted(counts.items())).encode())
    hsh.update(np.ascontiguousarray(p).tobytes())
    hsh.update(repr(float(delta)).encode())
    mine = hsh.hexdigest()
    if world == 1:
        return True
    got = [None] * world
    dist.all_gather_object(got, mine)
    return all(g == got[0] for g in got)


DUMP_BYTES = 64 << 20


def dump_outputs(dirname, arrays, limit=DUMP_BYTES):
    """Write every array as dirname/<name>.npy in float64, at most `limit` bytes in all.  Integer arrays (sampled keys)
    must be below 2^53 so that float64 holds them exactly.  An array too large for its share of the limit is replaced by
    its entries at a fixed, seeded sample of positions, which go to <name>_index.npy."""
    cap = limit // (8 * 2 * len(arrays))
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a).reshape(-1)
        if a.dtype.kind in 'iu' and a.size and int(a.max()) >= 1 << 53:
            raise ValueError('%s: integer values >= 2^53 have no exact float64 form' % name)
        a = a.astype(np.float64)
        if a.size > cap:
            idx = np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))
            np.save(os.path.join(dirname, name + '_index.npy'), idx.astype(np.float64))
            a = a[idx]
        np.save(os.path.join(dirname, name + '.npy'), a)


def workload_config(args, cliques, N):
    n = max(max(c) for c in cliques) + 1
    return {'workload': '%s: synthetic random-tree MRF, n=%d variables, k=%d pair cliques, N=%d total qubits, '
                        'complex64, %d shots + exact post-selected pmf per circuit' % (args.workload, n, len(cliques), N, SHOTS),
            'total_qubits': N, 'variables': n, 'cliques': len(cliques), 'shots': SHOTS,
            'l2': 'state (>= 8 GiB per GPU) far exceeds the 126 MB L2; no flush needed'}


# ------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='q34')
    ap.add_argument('--block-max', type=int, default=4)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-dense', action='store_true', help='skip the dense in-place gate-pass measurement')
    ap.add_argument('--dense-workload', default='q33')
    ap.add_argument('--dense-only', action='store_true', help='tuning aid: only the dense schedule, prints its dict')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last step of each timed arm returned as DIR/<name>.npy '
                         '(float64), so that two builds can be compared output for output')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'b200' or args.dense_only or args.workload in ('fixtures', 'chain20')):
        ap.error('--dump-outputs is implemented for the single-circuit workloads of --impl b200 only')
    if args.warmup < 3 and args.impl == 'b200':
        args.warmup = 3

    from qcmrf_b200 import workloads
    cliques, N = ([[0]], 3) if args.workload == 'fixtures' else workloads.named(args.workload)
    if args.impl == 'reference':
        run_reference_arm(args, cliques, N)
        return

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit('bench.py --gpus %d must be launched with torch.distributed.run (one rank per GPU)' % args.gpus)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device; qcmrf_b200 has no CPU path (use --impl reference for the CPU arm)')
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    from qcmrf_b200 import QCMRF, B200Simulator
    if world > 1:
        from qcmrf_b200.sharded import ShardedSimulator
        sim = ShardedSimulator(precision='single', block_max=args.block_max, device=local_rank, seed=1984)
    else:
        sim = B200Simulator(precision='single', fusion='blocked', block_max=args.block_max, device=local_rank,
                            seed=1984, small_batch=False)
    if args.workload == 'fixtures':
        sim.close()
        fixtures_bench(args, world, rank, local_rank, barrier_factory(torch, dist if world > 1 else None, world), torch,
                       dist if world > 1 else None)
        return
    if args.workload == 'chain20':
        sim.close()
        sweep_bench(args, world, rank, local_rank, barrier_factory(torch, dist if world > 1 else None, world), torch,
                    dist if world > 1 else None)
        return
    if args.dense_only:
        sim.close()
        d = dense_gate_pass(args, cliques, local_rank, world)
        if rank == 0:
            print(json.dumps(d), flush=True)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    thetas = [workloads.theta_for(cliques, seed=1984 + i) for i in range(args.warmup + args.steps + 2)]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- device-timed arm: planned program resident, tables on the host -----------------
    circ = QCMRF(cliques, thetas[0])
    prep = sim.prepare(circ)
    n_vars = prep.n_vars
    # warm-up: one blocking execution (its per-launch record is the fallback of the roofline entry), the rest through the
    # pipelined call of the timed loop, so that its one-time work (page-locked ring buffers, the device-side total, the
    # mark events) is not inside the timed region
    out = sim.execute(prep, SHOTS, seed=1984, stream=0)          # cold: module load, first-touch allocations
    out = sim.execute(prep, SHOTS, seed=1984, stream=0)
    # per-launch record (CUDA events inside the library) of the second (warm) blocking execution: the timed loop of a
    # sharded run only enqueues its programs, which leaves no per-op timings behind
    prof = sim.op_profile()
    kernels = sim.op_kernels() if hasattr(sim, 'op_kernels') else []
    for _ in range(args.warmup - 2):
        out = sim.execute_deferred(prep, SHOTS, seed=1984, stream=0)()
    launches0 = sim.kernel_launches()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    barrier()
    c_lo = clocks.mark()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    ev0.record()
    pending = None
    for _ in range(args.steps):
        # a stream of circuits: circuit i's read-back (and, sharded, its collective and key merge) is finished while
        # circuit i+1's gate program runs -- every result is collected inside the timed region
        fin = sim.execute_deferred(prep, SHOTS, seed=1984, stream=0)
        if pending is not None:
            out = pending()
        pending = fin
    if pending is not None:
        out = pending()
    ev1.record()
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    dev_ms = ev0.elapsed_time(ev1)
    launches = sim.kernel_launches() - launches0
    prof_source = 'second warm-up execution (blocking; CUDA events around every launch inside the library)'
    if world == 1:
        # the per-launch CUDA events of the LAST TIMED step (recorded inside the pipelined stream, read after the loop)
        try:
            pt = sim.op_profile()
            if len(pt) == len(prof) and max(r[1] for r in pt) > 0:
                prof = pt
                prof_source = 'last timed step (CUDA events around every launch inside the library, read after the timed loop)'
        except Exception:
            pass
    ms = torch.tensor([max(dev_ms, 0.0), wall_ms], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    dev_ms, wall_ms = (float(x) for x in ms.cpu())
    ms_per_step = dev_ms / args.steps

    # ---- end-to-end arm: the public call, host objects in, host results out ------------
    # the public call on a LIST of circuits, as the reference submits them (run_experiment.py:56: one run() for all
    # circuits): fresh theta per circuit, Philox stream = position in the list; the backend pipelines the list
    # (B200Simulator.run / ShardedSimulator.run): circuit i+1 is prepared and enqueued while circuit i's counts dict
    # is built.  Every circuit's tables go up and its keys + pmf come down inside the timed region.
    ths = [thetas[args.warmup + i + 1] for i in range(args.steps)]
    barrier()
    t1 = time.perf_counter()
    res = sim.run([QCMRF(cliques, t_) for t_ in ths], shots=SHOTS, seed=1984).result()
    counts_all = res.get_counts()
    pd = [res.postselected_probabilities(i) for i in range(args.steps)]
    torch.cuda.synchronize()
    e2e_ms = [(time.perf_counter() - t1) * 1e3 / args.steps]
    th, counts, (p, delta) = ths[-1], counts_all[-1], pd[-1]
    meta = res.metadata(args.steps - 1)
    h2d, d2h = meta.get('h2d_bytes', 0), meta.get('d2h_bytes', 0)
    # one more circuit through the blocking single-circuit call (what round 1 timed), for the line's e2e.single_ms
    barrier()
    t1 = time.perf_counter()
    res1 = sim.run(QCMRF(cliques, thetas[0]), shots=SHOTS, seed=7).result()
    res1.get_counts()
    res1.postselected_probabilities(0)
    single_ms = (time.perf_counter() - t1) * 1e3
    c_hi = clocks.mark()
    e2e_t = torch.tensor([float(np.mean(e2e_ms)), single_ms], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_ms_mean, single_ms = (float(x) for x in e2e_t.cpu())
    clk = clocks.stop(c_lo, c_hi) if rank == 0 else None
    same = ranks_identical(dist if world > 1 else None, world, counts, p, delta)
    if args.dump_outputs and rank == 0:
        # device-timed arm: (sampled keys, post-selected pmf, success probability) of its last step; e2e arm: the last
        # circuit of the list -- its pmf, success probability and counts (keys ascending)
        ck = sorted((int(k, 2), v) for k, v in counts.items())
        dump_outputs(args.dump_outputs, {'keys': out[0], 'pmf': out[1], 'delta': [out[2]], 'e2e_pmf': p, 'e2e_delta': [delta],
                                         'e2e_count_keys': [k for k, _ in ck], 'e2e_counts': [v for _, v in ck]})
    last_timing = sim.last_timing() if hasattr(sim, 'last_timing') else None
    breakdown = getattr(sim, 'breakdown_ms', None)
    dense = None
    if not args.no_dense:
        sim.close()
        try:
            dense = dense_gate_pass(args, cliques, local_rank, world)
        except Exception as e:                              # a secondary measurement must not cost the bench line
            dense = {'error': repr(e)[:500]}

    if rank == 0:
        peak, peak_src = load_peaks()
        # dominant launch of one program
        top = max(prof, key=lambda r: r[1])
        kind, top_ms, rd, wr = top
        # the dominant launch is the last pass of the program; its kernel name comes from the engine
        kname = (kernels[-1] if kernels and prof.index(top) == len(prof) - 1 and kernels[-1] else 'op kind %d' % kind)
        achieved = (rd + wr) / (top_ms * 1e-3) / 1e9
        total_bytes = sum(r[2] + r[3] for r in prof)
        prog_ms = sum(r[1] for r in prof)
        line = {'metric': METRIC, 'value': 1e3 / ms_per_step, 'unit': 'circuits/s', 'n_gpus': world,
                'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_per_step, 'higher_is_better': True,
                'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
                'config': workload_config(args, cliques, N),
                'clocks': clk,
                'e2e': {'value': 1e3 / e2e_ms_mean, 'unit': 'circuits/s', 'h2d_bytes_per_step': int(h2d),
                        'd2h_bytes_per_step': int(d2h), 'ms_per_step': e2e_ms_mean,
                        'what': 'one public run() call on the list of %d circuits (fresh theta each), pipelined by the backend; '
                                'time / circuits' % args.steps,
                        'single_circuit_call_ms': single_ms},
                'gpu_launches': int(launches),
                'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                             'traffic': ncu_traffic(args.workload, world)[0], 'peak_source': peak_src,
                             'launch_ms_source': prof_source,
                             'traffic_source': '%s (ncu --set full of this kernel, same workload, 1 GPU)' % ncu_traffic(args.workload, world)[1],
                             'kernel': '%s: reads %d B, writes %d B in %.3f ms' % (kname, rd, wr, top_ms)},
                'program': {'passes': [{'kind': r[0], 'ms': r[1], 'read': r[2], 'written': r[3],
                                        'gbs': (r[2] + r[3]) / max(r[1], 1e-9) / 1e6} for r in prof],
                            'program_ms': prog_ms, 'program_gbs': total_bytes / max(prog_ms, 1e-9) / 1e6,
                            'wall_ms_per_step': wall_ms / args.steps},
                'hbm_gbs_program': total_bytes / max(prog_ms, 1e-9) / 1e6,
                'device_timing_last_step': last_timing, 'host_breakdown_ms': breakdown, 'dense_gate_pass': dense,
                'check': dict({'delta': float(delta), 'p_sum': float(np.sum(p)), 'shots': int(sum(counts.values())),
                               'ranks_identical': bool(same)},
                              **parity_check(cliques, th, p, delta, counts)),
                'value_note': 'the device-timed arm re-executes one prepared circuit (same theta, seed and Philox stream) '
                              'every step; e2e uses a fresh theta per circuit.  Both arms, at every N, run the circuits as a '
                              'pipeline (execute_deferred / run(list)): programs and result handling are enqueued, every '
                              'result is collected inside the timed region; e2e.single_circuit_call_ms is one blocking '
                              'run() on a single circuit'}
        if world == 1 and not args.no_cpu_baseline:
            line['cpu_baseline'], _ = cpu_reference(cliques, steps=1, warmup=0)
        print(json.dumps(line), flush=True)
    try:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        sim.close()
    except Exception as e:
        print('bench.py: teardown: %r' % (e,), file=sys.stderr)


def barrier_factory(torch, dist, world):
    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
    return barrier


def fixtures_bench(args, world, rank, device, barrier, torch, dist):
    """BASELINE config 1: all 210 res_0.1 / res_0.25 / res_0.5 fixture models in one batch -- exact
    post-selected pmf + 8192 shots each -- through the batched small-circuit kernel (one CTA per circuit,
    one launch), complex128.  With N GPUs the list is split round-robin, no communication."""
    from qcmrf_b200 import QCMRF, B200Simulator
    models = json.load(open(os.path.join(ROOT, 'tests', 'golden', 'models.json')))
    items = [(C, th) for sc in ('0.1', '0.25', '0.5') for j, C in enumerate(models[sc]['GRAPHS'])
             for th in models[sc]['THETAS'][str(j)]]
    mine = list(range(rank, len(items), world))
    shots = 8192
    sim = B200Simulator(precision='double', device=device, seed=1984)
    times, dev = [], []
    for it in range(args.warmup + args.steps):
        barrier()
        t0 = time.perf_counter()
        res = sim.run([QCMRF(*items[i]) for i in mine], shots=shots, stream_ids=mine).result()
        counts = res.get_counts()
        torch.cuda.synchronize()
        if it >= args.warmup:
            times.append((time.perf_counter() - t0) * 1e3)
            dev.append(res.metadata(0)['batch_device_ms'])
    red = torch.tensor([float(np.mean(times)), float(np.mean(dev))], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(red, op=dist.ReduceOp.MAX)
    e2e_ms, dev_ms = (float(x) for x in red.cpu())
    # the reference's literal flow (run_experiment.py:44-57) on its own 70 models of one scale: construct, transpile to
    # cx/id/rz/sx/x, run(T, shots=10000), get_counts -- the transpiled circuits (up to ~15 000 basis gates each) must be
    # fused back into one sweep per clique by the gate-fusion pass before they reach the GPU
    ref_flow = None
    if rank == 0:
        from qcmrf_b200 import transpile
        flow = []
        for it in range(3):
            t0 = time.perf_counter()
            CIRCS = [QCMRF(C, th, with_measurements=True) for C, th in items[140:210]]          # res_0.5
            t1 = time.perf_counter()
            T = transpile(CIRCS, basis_gates=['cx', 'id', 'rz', 'sx', 'x'])
            t2 = time.perf_counter()
            result = sim.run(T, shots=10000).result()
            t3 = time.perf_counter()
            cts = result.get_counts()
            torch.cuda.synchronize()
            t4 = time.perf_counter()
            flow.append([(t1 - t0) * 1e3, (t2 - t1) * 1e3, (t3 - t2) * 1e3, (t4 - t3) * 1e3, (t4 - t0) * 1e3])
        best = min(flow, key=lambda r: r[-1])
        gates = sum(len(T[k]._lower_program().bk) for k in range(len(T)))
        ref_flow = {'circuits': len(CIRCS), 'basis_gates_total': int(gates), 'construct_ms': best[0], 'transpile_ms': best[1],
                    'run_ms (lower + gate fusion + plan + one batched launch + counts dicts)': best[2], 'get_counts_ms': best[3],
                    'total_ms': best[4], 'ms_per_circuit': best[4] / len(CIRCS), 'shots': 10000,
                    'check_shots': int(sum(cts[0].values()))}
    if rank == 0:
        n = len(items)
        line = {'metric': METRIC, 'value': n / (dev_ms * 1e-3), 'unit': 'circuits/s', 'n_gpus': world, 'steps': args.steps,
                'warmup': args.warmup, 'ms_per_step': dev_ms, 'higher_is_better': True, 'scaling': 'strong',
                'vs_baseline': None, 'dtype': 'f64', 'data': 'reference fixtures (res_*/models*.json)',
                'config': {'workload': 'fixtures: the 210 models of res_0.1/res_0.25/res_0.5 (3..10 qubits), one batch, exact pmf + '
                                       '8192 shots each, complex128', 'circuits': n, 'shots': shots,
                           'l2': 'states live in shared memory (<= 16 KiB each): latency-bound single launch'},
                'e2e': {'value': n / (e2e_ms * 1e-3), 'unit': 'circuits/s', 'ms_per_step': e2e_ms,
                        'h2d_bytes_per_step': None, 'd2h_bytes_per_step': int(len(mine) * shots * 8)},
                'gpu_launches': args.steps,
                'note': 'value = the single k_small launch (CUDA events inside the library); e2e = B200Simulator.run(list of '
                        'QCMRF objects) -> counts dicts + pmfs, dominated by host-side lowering/fusion and key formatting',
                'reference_flow': ref_flow,
                'check': {'shots': int(sum(counts[0].values())), 'n_results': len(counts)}}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    sim.close()


def sweep_bench(args, world, rank, device, barrier, torch, dist):
    """BASELINE config 3: 20-variable chain MRF, complex128, 256-point beta-sweep (beta_j = (j+1)/128, QCMRF.py:21,154),
    the points partitioned round-robin over the GPUs with no communication.  At Aer width the circuit has 40 qubits
    (16 TiB); it is run measure-and-release (width='release'): the 20 variable qubits are stored (16 MiB per point),
    every clique ancilla is drawn from its sweep's coefficients and projected for the exact post-selected pmf.
    All points of a rank go through ONE batched handle: every kernel is launched once for the whole sweep
    (qcm_create_batched).  A step = the whole sweep: 256 circuits, each with delta, its 2^20 pmf (left on the GPU
    unless asked for) and 10000 full-width (40-bit) shots."""
    from qcmrf_b200 import QCMRF, B200Simulator, workloads
    points = 256
    cliques, N = workloads.named('chain20')
    n = 20
    theta = workloads.theta_for(cliques)
    betas = [(j + 1) / 128.0 for j in range(points)]
    mine = list(range(rank, points, world))
    sim = B200Simulator(precision='double', width='release', device=device, seed=1984, small_batch=False)
    sw = sim.prepare_sweep([QCMRF(cliques, theta, beta=betas[j]) for j in mine])
    streams = np.asarray(mine, dtype=np.uint64)
    for _ in range(args.warmup):
        sim.execute_sweep(sw, SHOTS, seed=1984, streams=streams)
    l0 = sim.kernel_launches()
    clocks = ClockSampler(device)
    if rank == 0:
        clocks.start()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        keys, probs, kept = sim.execute_sweep(sw, SHOTS, seed=1984, streams=streams)
    ev1.record()
    barrier()
    dev_ms = ev0.elapsed_time(ev1)
    launches = sim.kernel_launches() - l0
    sim.execute_sweep(sw, SHOTS, seed=1984, streams=streams, profile=True)      # untimed: the per-launch record
    prof = sim.sweep_profile
    e2e, e2e_keys = [], []
    for i in range(args.steps):
        barrier()
        t1 = time.perf_counter()
        res = sim.run([QCMRF(cliques, theta, beta=betas[j]) for j in mine], shots=SHOTS, seed=1984 + i, stream_ids=mine).result()
        deltas = [res.success_probability(k) for k in range(len(mine))]
        counts = res.get_counts()
        torch.cuda.synchronize()
        e2e.append((time.perf_counter() - t1) * 1e3)
    m = res.metadata(0)
    red = torch.tensor([dev_ms, float(np.mean(e2e))], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(red, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms = (float(x) for x in red.cpu())
    clk = clocks.stop() if rank == 0 else None
    # parity of this rank's first / middle / last point against brute-force enumeration (2^20 states)
    chk = {}
    for k in sorted({0, len(mine) // 2, len(mine) - 1}):
        p, d = res.postselected_probabilities(k)
        c = parity_check(cliques, theta, p, d, counts[k], beta=betas[mine[k]], tol=1e-10, rel_tol=1e-9)
        chk['beta=%g' % betas[mine[k]]] = {kk: c[kk] for kk in ('max_abs_p_error_vs_brute_force', 'rel_p_err', 'delta_rel_err', 'tv',
                                                               'tv_bound', 'sampled_success_fraction', 'exact_delta', 'parity_ok')}
    ok = all(v['parity_ok'] for v in chk.values())
    oks = [None] * world
    if world > 1:
        dist.all_gather_object(oks, ok)
    else:
        oks = [ok]
    if rank == 0:
        peak, peak_src = load_peaks()
        ms_step = dev_ms / args.steps
        launches_all = prof['program'] + prof['projection']
        top = max(launches_all, key=lambda r: r[1][1])
        top_name, (_kind, top_ms, top_rd, top_wr) = top
        amp = 16 << n
        B = len(mine)
        tree_read = B * amp if os.environ.get('QCM_PRODUCT_SAMPLE') == '0' else 0
        algo = (sum(r[1][2] + r[1][3] for r in launches_all)      # init write + the projection passes
                + tree_read                                        # sampler: the stored state of an all-released QCMRF is a
                                                                   # product state, drawn per qubit (no sum tree, no state read)
                + B * amp + B * (8 << n))                          # post-selection: read the state, write the pmf
        line = {'metric': METRIC, 'value': points / (ms_step * 1e-3), 'unit': 'circuits/s', 'n_gpus': world,
                'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_step, 'higher_is_better': True,
                'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
                'config': {'workload': 'chain20: 20-variable chain MRF (k=19, N=40 qubits at Aer width), complex128, '
                                       '256-point beta-sweep, measure-and-release width (20 stored qubits), %d shots + delta + exact '
                                       'pmf (device-resident) per point; one batched handle per GPU' % SHOTS, 'points': points,
                           'points_per_gpu': B, 'stored_qubits': m['n_phys'], 'released_qubits': m['released_qubits'], 'shots': SHOTS,
                           'l2': 'the %d states of a rank are %.1f GiB in one allocation, swept by every kernel: far beyond the 126 MB L2'
                                 % (B, B * amp / 2.0 ** 30)},
                'clocks': clk,
                'e2e': {'value': points / (e2e_ms * 1e-3), 'unit': 'circuits/s', 'ms_per_step': e2e_ms,
                        'h2d_bytes_per_step': int(m['h2d_bytes']) * B, 'd2h_bytes_per_step': int(m['d2h_bytes']) * B,
                        'what': 'B200Simulator.run(list of 256 QCMRF objects) -> counts dicts (40-bit keys) + delta of every point; '
                                'pmfs stay on the GPU until asked for'},
                'gpu_launches': int(launches),
                'roofline': {'bound': 'hbm', 'achieved': (top_rd + top_wr) / (top_ms * 1e-3) / 1e9, 'peak': peak, 'unit': 'GB/s',
                             'frac': (top_rd + top_wr) / (top_ms * 1e-3) / 1e9 / peak, 'traffic': None, 'peak_source': peak_src,
                             'kernel': '%s over %d states at once: reads %d B, writes %d B in %.3f ms' % (top_name or 'op', B, top_rd, top_wr, top_ms)},
                'sweep': {'launches_per_sweep': int(launches) // max(args.steps, 1), 'algorithmic_bytes_per_sweep': int(algo),
                          'hbm_gbs_whole_sweep': algo / (ms_step * 1e-3) / 1e9, 'frac_of_peak_whole_sweep': algo / (ms_step * 1e-3) / 1e9 / peak,
                          'passes': [{'kernel': nm, 'ms': r[1], 'gbs': (r[2] + r[3]) / max(r[1], 1e-9) / 1e6} for nm, r in launches_all],
                          'sample_ms': prof['sample_ms'], 'postselect_ms': prof['postselect_ms'],
                          'host_wall_ms_program_shots_projection_postselect': prof.get('host_wall_ms')},
                'check': dict({'points_checked_vs_brute_force': chk, 'all_ranks_ok': bool(all(oks)),
                               'shots': int(sum(counts[-1].values())), 'delta_first_last': [deltas[0], deltas[-1]]})}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    sim.close()


def dense_gate_pass(args, cliques, device, world=1):
    """The plain in-place gate pass (one fused clique = one read+write sweep of the whole,
    fully materialised state): the kernel BASELINE.json's 70%-of-roofline target is about.
    Not the product's default schedule -- the lazily materialised one above moves ~30x fewer
    bytes per circuit.  Sharded (world > 1): canonical layout, the last log2(world) clique
    ancillas are global and come on-GPU through ONE qubit-swap all-to-all (NCCL send/recv
    over NVLink), which is timed here."""
    from qcmrf_b200 import QCMRF, B200Simulator, workloads
    peak, _ = load_peaks()
    cliques, _ = workloads.named(args.dense_workload)   # q33: 33 physical qubits = 64 GiB in total, identity layout
    circ = QCMRF(cliques, workloads.theta_for(cliques))
    if world == 1:
        sim = B200Simulator(precision='single', fusion='clique', device=device, seed=1, small_batch=False)
    else:
        from qcmrf_b200.sharded import ShardedSimulator
        sim = ShardedSimulator(precision='single', fusion='clique', layout='canonical', device=device, seed=1,
                               staging_bytes=2 << 30)
        sim.sync_before_exchange = True
    prep = sim.prepare(circ)
    sim.execute(prep, 0, want_probs=False)
    sim.execute(prep, 0, want_probs=False)
    prof = sim.op_profile()
    passes = [r for r in prof if r[0] == 2 and r[2] == r[3] and r[2] > 0]
    ms = float(np.median([r[1] for r in passes]))
    by = passes[0][2] + passes[0][3]
    out = {'workload': '%s, fusion=clique: one in-place pass per clique' % args.dense_workload, 'n_phys': prep.plan.n_phys,
           'ranks': world, 'passes': len(passes), 'bytes_per_pass_per_gpu': by, 'median_ms': ms,
           'gbs_per_gpu': by / ms / 1e6, 'frac_of_measured_peak': by / ms / 1e6 / peak,
           'amp_updates_per_sec_all_gpus': world * (by / 16) / (ms * 1e-3), 'circuit_ms': sum(r[1] for r in prof),
           'init_ms': [r[1] for r in prof if r[0] == 1][0], 'init_gbs': [r[3] / r[1] / 1e6 for r in prof if r[0] == 1][0]}
    ex = [r for r in prof if r[0] == -1]
    if ex:
        out['exchange'] = [{'ms': r[1], 'bytes_sent_per_gpu': r[2], 'gbs_per_direction_per_gpu': r[2] / r[1] / 1e6}
                           for r in ex]
    sim.close()
    # the same schedule with the qubit swap and the sweeps on the swapped-in qubits fused into ONE kernel that reads the
    # peers' shards over NVLink: out of place (a second local buffer: shards <= 32 GiB here) and IN PLACE (per-tile
    # flags order the overwrites behind the peers' reads: any shard size, e.g. the 128 GiB shards of 37 qubits on 8 GPUs)
    s = world.bit_length() - 1
    variants = []
    if world > 1 and prep.plan.n_phys - s <= 32:
        variants.append(('fused_exchange', 'p2p'))
    if world > 1:
        variants.append(('fused_exchange_inplace', 'p2p-inplace'))
    for key, xch in variants:
        from qcmrf_b200.sharded import ShardedSimulator
        sim = ShardedSimulator(precision='single', fusion='clique', layout='canonical', device=device, seed=1, exchange=xch)
        prep = sim.prepare(circ)
        try:
            sim.execute(prep, 0, want_probs=False)
            res2 = sim.execute(prep, 0, want_probs=True)
        except Exception as e:
            out[key] = {'error': repr(e)[:500]}
            try:
                sim.close()
            except Exception:
                pass
            continue
        prof2 = sim.op_profile()
        fx = [r for r in prof2 if r[0] == -2]
        if fx:
            remote = fx[0][2] * (world - 1) // world        # every output pair takes 2^s inputs, all but one from peers
            out[key] = {'kernel': '%s: qubit swap + the %d sweeps on the swapped-in qubits, peers read over NVLink (CUDA IPC, TMA '
                                  'bulk copies into a shared-memory ring)' % ('k_block_gather_inplace' if xch == 'p2p-inplace' else
                                                                             'k_block_gather_tma', s),
                        'ms': fx[0][1], 'replaces_ms': (ex[0][1] if ex else 0.0) + s * ms,
                        'remote_bytes_read_per_gpu': remote, 'nvlink_gbs_per_gpu': remote / fx[0][1] / 1e6,
                        'circuit_ms': sum(r[1] for r in prof2)}
            n_v = max(max(c) for c in cliques) + 1
            if res2[1] is not None and n_v <= 24:
                pb, db = brute_force_pmf(cliques, workloads.theta_for(cliques))
                p2 = res2[1] / res2[2]
                out[key]['check'] = {'rel_p_err_vs_brute_force': float((np.abs(p2 - pb) / pb).max()),
                                     'delta_rel_err': abs(float(res2[2]) - db) / db,
                                     'parity_ok': bool((np.abs(p2 - pb) / pb).max() < 2e-4 and abs(float(res2[2]) - db) / db < 2e-4)}
        else:
            out[key] = {'unavailable': getattr(sim, 'p2p_error', 'no fused segment in the plan')}
        sim.close()
    return out


if __name__ == '__main__':
    main()
