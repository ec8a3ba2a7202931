"""Noisy-shot throughput on one GPU: the reference's 70 transpiled fixture circuits of one scale under depolarizing
gate errors and readout errors, and under a hardware-like model with thermal relaxation.

Workload: scale 0.5 (7 graphs x 10 thetas, 3-10 qubits, 47-14 708 gates), 10^4 shots each, 2 % symmetric readout
error and one of two gate-error models:
  * Pauli-only: depolarizing p1 = 1e-3 after sx / x / id, p2 = 1e-2 after cx (qcm_run_noisy_small);
  * hardware-like (what NoiseModel.from_backend builds in Aer): depolarizing p1 = 1e-3 composed with
    thermal_relaxation_error(100 us, 80 us, 35.5 ns) after sx / x / id, p2 = 1e-2 composed with two 300 ns
    relaxations expanded over the qubits after cx; nothing after the virtual rz (qcm_run_noisy_small_kraus).
It reports, per precision, the device time of each trajectory launch (CUDA events around the entry's kernels),
trajectories/s and gate applications/s; the Pauli-only workload once more through qcm_run_noisy_small_kraus (its
channels as one-stage error records), which prices keeping the Pauli-only entry; the device time of the
readout-only route (the ideal batched kernel plus k_readout_keys) next to the ideal batched kernel alone; and the
wall time of the whole B200Simulator.run() call.  Prints one JSON line; reads the card's name and power limit in
the same run.

    python tools/noise_bench.py [--shots 10000] [--reps 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from qcmrf_b200 import QCMRF, B200Simulator, _native, ir, transpile  # noqa: E402
from qcmrf_b200.noise import (NoiseModel, ReadoutError, depolarizing_error, encode,  # noqa: E402
                              thermal_relaxation_error)


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, power = [x.strip() for x in out[0].split(',')]
        return {'gpu': name, 'power_limit': power}
    except Exception as e:                                  # the numbers still stand; say what is missing
        return {'gpu': None, 'power_limit': None, 'card_query_error': str(e)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--shots', type=int, default=10000)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--scale', default='0.5')
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    if _native.device_count() < 1:
        raise SystemExit('noise_bench: no CUDA device')
    models = json.load(open(os.path.join(ROOT, 'tests', 'golden', 'models.json')))
    circs = []
    for j, C in enumerate(models[a.scale]['GRAPHS']):
        for th in models[a.scale]['THETAS'][str(j)]:
            circs.append(transpile([QCMRF(C, th)], basis_gates=['cx', 'id', 'rz', 'sx', 'x'])[0])
    nm = NoiseModel()
    nm.add_all_qubit_quantum_error(depolarizing_error(1e-3, 1), ['sx', 'x', 'id'])
    nm.add_all_qubit_quantum_error(depolarizing_error(1e-2, 2), ['cx'])
    nm.add_all_qubit_readout_error(ReadoutError([[0.98, 0.02], [0.02, 0.98]]))
    hw = NoiseModel()
    t1q, t2q = thermal_relaxation_error(100e-6, 80e-6, 35.5e-9), thermal_relaxation_error(100e-6, 80e-6, 300e-9)
    hw.add_all_qubit_quantum_error(depolarizing_error(1e-3, 1).compose(t1q), ['sx', 'x', 'id'])
    hw.add_all_qubit_quantum_error(depolarizing_error(1e-2, 2).compose(t2q.expand(t2q)), ['cx'])
    hw.add_all_qubit_readout_error(ReadoutError([[0.98, 0.02], [0.02, 0.98]]))
    ro_only = NoiseModel()
    ro_only.add_all_qubit_readout_error(ReadoutError([[0.98, 0.02], [0.02, 0.98]]))
    progs = [ir.lower(c) for c in circs]
    t0 = time.perf_counter()
    enc = [encode(p, nm) for p in progs]
    encode_ms = (time.perf_counter() - t0) * 1e3
    t0 = time.perf_counter()
    enc_hw = [encode(p, hw) for p in progs]
    encode_hw_ms = (time.perf_counter() - t0) * 1e3
    assert all(e.kraus for e in enc_hw) and not any(e.kraus for e in enc)
    gates = int(sum(e.n_gates for e in enc))
    traj = len(enc) * a.shots
    out = dict(card(), workload={'circuits': len(enc), 'scale': a.scale, 'shots': a.shots, 'gates': gates,
                                 'qubits': [int(min(p.n_qubits for p in progs)), int(max(p.n_qubits for p in progs))],
                                 'p1': 1e-3, 'p2': 1e-2, 'readout': 0.02,
                                 'hardware_like': {'t1': 100e-6, 't2': 80e-6, 'time_1q': 35.5e-9, 'time_cx': 300e-9,
                                                   'gates_with_error': int(sum((e.channel >= 0).sum() for e in enc_hw)),
                                                   'kraus_stages_per_circuit_max': int(max(len(e.kraus_n_ops) for e in enc_hw))}},
               host_encode_ms=round(encode_ms, 2), host_encode_hw_ms=round(encode_hw_ms, 2), reps=a.reps)
    for precision in ('double', 'single'):
        r = {}
        arms = (('pauli_only', _native.run_noisy_small, enc), ('hardware_like', _native.run_noisy_small_kraus, enc_hw),
                ('pauli_only_via_kraus_entry', _native.run_noisy_small_kraus, enc))
        for name, run, e in arms:
            run(e, a.shots, 1, precision=precision)                                  # warm-up
        ms = {name: [] for name, _, _ in arms}
        for k in range(a.reps):                                   # the arms alternate, so drift hits all alike
            for name, run, e in arms:
                ms[name].append(run(e, a.shots, 100 + k, precision=precision)[1])
        for name, _, _ in arms:
            t = float(np.median(ms[name]))
            r[name] = {'trajectory_launch_ms': round(t, 3),
                       'trajectory_launch_ms_min_max': [round(min(ms[name]), 3), round(max(ms[name]), 3)],
                       'trajectories_per_s': traj / (t * 1e-3), 'gate_applications_per_s': gates * a.shots / (t * 1e-3)}
        sim = B200Simulator(precision=precision, seed=7)
        prs = [sim.prepare(p, small=True) for p in progs]
        args = ([pr.plan for pr in prs], [pr.clbit_map for pr in prs], [(0, 0, 0)] * len(prs), a.shots, 3)
        ro = np.stack([e.readout for e in enc])
        for key, kw in (('ideal_batch_small_ms', {}), ('readout_only_route_ms', {'readout': ro})):
            _native.run_batch_small(*args, precision=precision, **kw)
            ms = [_native.run_batch_small(*args, precision=precision, **kw)[3] for _ in range(a.reps)]
            r[key] = round(float(np.median(ms)), 4)
        for key, model in (('run_wall_ms_noisy', nm), ('run_wall_ms_hardware_like', hw),
                           ('run_wall_ms_readout_only', ro_only)):
            sim.run(circs, shots=a.shots, noise_model=model).result()
            w = []
            for _ in range(a.reps):
                t0 = time.perf_counter()
                sim.run(circs, shots=a.shots, noise_model=model).result()
                w.append((time.perf_counter() - t0) * 1e3)
            r[key] = round(float(np.median(w)), 2)
        out[precision] = r
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
