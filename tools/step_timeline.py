"""Where one step of the flagship workload's time goes: the q34 pipelined loop of bench.py's device-timed arm
(execute_deferred, steps back to back) under torch.profiler with CUDA activities.

    python tools/step_timeline.py --out DIR [--steps 30] [--warmup 5]

Writes DIR/step_timeline.pt.trace.json (the raw trace) and DIR/step_timeline.json:
  - the device events (kernels, copies, memsets) of one steady-state step, each with its duration and the gap before it;
  - the step period (start to start on the device), the device busy time, and the gaps' sum;
  - the host time per step spent enqueuing (run_program, sample, postselect, mark) and collecting, the latter split into
    waiting for the device (wait) and the host's own work (result copies);
  - the card's name and power limit.
Run it alone: tracing slows the host, so its step period is not the benchmark's.

    python tools/step_timeline.py --out DIR --no-profiler [--steps 200] [--warmup 5]

runs the same loop without the profiler and writes DIR/step_host.json: per step, the host clock around the enqueue
(execute_deferred) and around the collect (the previous circuit's callable), their medians, the host time per engine
call, and the loop's wall time per step.  When enqueue + collect minus the wait is close to the wall time per step, the
host is the limit; otherwise the device is.
"""
import argparse
import collections
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

SHOTS = 10000


def _card():
    try:
        return subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                    # the number still stands; say what is missing
        return 'unknown (%s)' % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--steps', type=int, default=30)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--no-profiler', action='store_true', help='host clocks only (see the module docstring)')
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    import torch
    from torch.profiler import ProfilerActivity, profile
    from qcmrf_b200 import QCMRF, B200Simulator, _native, workloads

    # host time per engine call, accumulated per step
    host = {}

    def timed(name, fn):
        def wrap(self, *a, **k):
            t0 = time.perf_counter()
            try:
                return fn(self, *a, **k)
            finally:
                host[name] = host.get(name, 0.0) + time.perf_counter() - t0
        return wrap

    for name in ('run_program', 'sample', 'postselect', 'mark', 'wait'):
        setattr(_native.Handle, name, timed(name, getattr(_native.Handle, name)))

    cliques, _ = workloads.named('q34')
    sim = B200Simulator(precision='single', fusion='blocked', block_max=4, seed=1984, small_batch=False)
    prep = sim.prepare(QCMRF(cliques, workloads.theta_for(cliques, seed=1984)))
    sim.execute(prep, SHOTS, seed=1984, stream=0)
    for _ in range(args.warmup):
        sim.execute_deferred(prep, SHOTS, seed=1984, stream=0)()
    torch.cuda.synchronize()
    host.clear()
    if args.no_profiler:
        host_only(args, sim, prep, host, torch)
        return
    enq = col = 0.0
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        pending = None
        for _ in range(args.steps):
            t0 = time.perf_counter()
            fin = sim.execute_deferred(prep, SHOTS, seed=1984, stream=0)
            t1 = time.perf_counter()
            enq += t1 - t0
            if pending is not None:
                pending()
            col += time.perf_counter() - t1
            pending = fin
        t1 = time.perf_counter()
        pending()
        col += time.perf_counter() - t1
        torch.cuda.synchronize()
    kernels = sim.op_kernels()
    sim.close()
    trace = os.path.join(args.out, 'step_timeline.pt.trace.json')
    prof.export_chrome_trace(trace)

    ev = [e for e in json.load(open(trace))['traceEvents']
          if e.get('ph') == 'X' and e.get('cat') in ('kernel', 'gpu_memcpy', 'gpu_memset')]
    ev.sort(key=lambda e: e['ts'])
    # a step starts with the earliest device event that runs once per step (the program's first kernel)
    once = collections.Counter(e['name'] for e in ev)
    first = next(e['name'] for e in ev if once[e['name']] == args.steps)
    starts = [i for i, e in enumerate(ev) if e['name'] == first]
    assert len(starts) == args.steps, (first, len(starts))
    steps = [ev[a:b] for a, b in zip(starts, starts[1:] + [len(ev)])]
    periods = [steps[k + 1][0]['ts'] - steps[k][0]['ts'] for k in range(len(steps) - 1)]
    busy = [sum(e['dur'] for e in s) for s in steps[:-1]]
    mid = len(steps) // 2
    prev_end = steps[mid - 1][-1]['ts'] + steps[mid - 1][-1]['dur']
    rows = []
    for e in steps[mid]:
        rows.append({'name': e['name'][:160], 'cat': e['cat'], 'dur_us': round(e['dur'], 2),
                     'gap_before_us': round(e['ts'] - prev_end, 2)})
        prev_end = e['ts'] + e['dur']
    n = args.steps
    host_ms = {k: round(v * 1e3 / n, 4) for k, v in sorted(host.items())}
    host_ms['enqueue (execute_deferred)'] = round(enq * 1e3 / n, 4)
    host_ms['collect (wait, result copies)'] = round(col * 1e3 / n, 4)
    period = float(np.median(periods)) / 1e3
    # the loop waits for step k-1 before it enqueues step k+1, so enqueue + collect always spans the device period; the
    # host bounds the step only when its work without the wait does
    work = (enq + col - host.get('wait', 0.0)) * 1e3 / n
    out = {
        'card': _card(),
        'workload': 'q34, complex64, 10^4 shots, execute_deferred back to back (profiler on)',
        'steps': n,
        'step_period_ms_median': round(period, 4),
        'device_busy_ms_median': round(float(np.median(busy)) / 1e3, 4),
        'device_idle_ms_median': round(period - float(np.median(busy)) / 1e3, 4),
        'host_ms_per_step': host_ms,
        'host_per_step_ms': round((enq + col) * 1e3 / n, 4),
        'host_work_per_step_ms': round(work, 4),
        'bound': 'host' if work >= 0.9 * period else 'gpu',
        'program_kernels': kernels,
        'step_index': mid,
        'events': rows,
    }
    with open(os.path.join(args.out, 'step_timeline.json'), 'w') as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ('card', 'step_period_ms_median', 'device_busy_ms_median',
                                          'device_idle_ms_median', 'host_work_per_step_ms', 'bound')}))


def host_only(args, sim, prep, host, torch):
    """The pipelined loop of bench.py's device-timed arm with host clocks around each step's enqueue and collect."""
    enq, col = [], []
    t_start = time.perf_counter()
    pending = None
    for _ in range(args.steps):
        t0 = time.perf_counter()
        fin = sim.execute_deferred(prep, SHOTS, seed=1984, stream=0)
        t1 = time.perf_counter()
        if pending is not None:
            pending()
        col.append(time.perf_counter() - t1)
        enq.append(t1 - t0)
        pending = fin
    t1 = time.perf_counter()
    pending()
    col[-1] += time.perf_counter() - t1
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t_start) * 1e3 / args.steps
    sim.op_profile()                                          # what bench.py reads after its loop
    sim.close()
    n = args.steps
    wait = host.get('wait', 0.0) * 1e3 / n
    ms = lambda v: round(float(v) * 1e3, 4)                   # noqa: E731
    out = {
        'card': _card(),
        'workload': 'q34, complex64, 10^4 shots, execute_deferred back to back (profiler off, host clocks)',
        'steps': n,
        'wall_ms_per_step': round(wall, 4),
        'enqueue_ms_median': ms(np.median(enq)),
        'collect_ms_median': ms(np.median(col)),
        'enqueue_ms_mean': ms(np.mean(enq)),
        'collect_ms_mean': ms(np.mean(col)),
        'host_ms_per_call': {k: round(v * 1e3 / n, 4) for k, v in sorted(host.items())},
        'host_work_per_step_ms': round((sum(enq) + sum(col)) * 1e3 / n - wait, 4),
    }
    out['bound'] = 'host' if out['host_work_per_step_ms'] >= 0.9 * wall else 'gpu'
    with open(os.path.join(args.out, 'step_host.json'), 'w') as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == '__main__':
    main()
