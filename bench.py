#!/usr/bin/env python
"""bench.py — benchmark of the hot path (see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl cuda|reference] [--workload NAME] [--replicas R] [--lpr L]
                    [--dump-outputs DIR]

Workloads (BASELINE.json configs; default fifo60k = the configuration the metric "simulated events/sec on 60k-job trace" is
quoted on and the only one with a measured reference number on that trace):
    fifo60k     fifo + yarn, 60 000-job trace gen(60000, seed, 60000), 4x32x8 simulated cluster        (C3-sized trace, live reference path)
    dlas60k     dlas-gpu (4-queue MLFQ, limits 30/60/150 GPU-ticks), same trace, admission by GPU count    (C3)
    sjf10k      sjf + yarn, 10 000-job trace gen(10000, seed, 10000)                                       (C2)
    env512x10k  512 environment replicas per GPU of 10 000-job traces, random-window policy rolled out on the device  (C4; --gpus 8 = C5)
One "step" = every replica of the GPU simulated to completion.  An event = arrival | start | finish | preemption | resume |
queue jump (SURVEY.md 8d); 3 per finished job under non-preemptive fifo.

Prints ONE JSON line (rank 0).  `value` = events/s with traces resident in HBM (rows written to the device-resident row
store); `e2e` = the same through the C ABI with host buffers: trace upload (records in pinned host memory), simulation, the result of every replica copied
back to the host, all inside the timed region.  For fifo the result is the per-tick row stream in `--rows-format`: event4
(default; 4 bytes per tick = the event log, from which rlgs_read_rows / rlgs_read_jobs rebuild every column and table of a
replica on demand), event16 (also reported as `e2e_stat_rows`: the rows still carry the kernel-computed pending statistics),
wire12 / wire16 (+ job tables), wide (the 64-byte rows of round 1).  `--impl reference` times the reference's algorithm on the host cores (oracle/cpu_sim.c, the
C port validated byte-for-byte against the real Python reference) and, when the unmodified Python reference was staged under
oracle/_ref/reference by __graft_entry__.build(), reports its own measured events/s beside it (`reference_python`).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CLUSTER_FLAGS = dict(num_switch=4, num_node_p_switch=32, num_gpu_p_node=8)
METRIC = 'simulated_events_per_sec'
UNIT = 'events/s'
REF_DIR = os.path.join(ROOT, 'oracle', '_ref', 'reference')

WORKLOADS = {
    'fifo60k': dict(schedule='fifo', scheme='yarn', n_jobs=60000, seed0=3, n_traces=16, replicas=8880, kw={},
                    text='fifo+yarn, 4x32x8 simulated cluster, 60k-job Philly-style trace (gen(60000, seed, 60000))'),
    'dlas60k': dict(schedule='dlas-gpu', scheme='count', n_jobs=60000, seed0=3, n_traces=8, replicas=4736,
                    kw=dict(num_queue=4, queue_limit=(30, 60, 150)),
                    text='dlas-gpu (4-queue MLFQ, limits 30/60/150 GPU-ticks), 4x32x8 simulated cluster, 60k-job trace (gen(60000, seed, 60000))'),
    'sjf10k': dict(schedule='sjf', scheme='yarn', n_jobs=10000, seed0=2, n_traces=8, replicas=4736, kw={},   # 64-register build: 32 warps per SM
                   text='sjf+yarn, 4x32x8 simulated cluster, 10k-job trace (gen(10000, seed, 10000))'),
    'env512x10k': dict(schedule='fifo', scheme='yarn', n_jobs=10000, seed0=1000, n_traces=32, replicas=512, kw={}, env=True,
                       text='RL environment rollouts (random pick inside a 5-job window, counter-based RNG), 4x32x8 simulated cluster, '
                            '10k-job traces (gen(10000, 1000 + i, 10000))'),
}


def frames(w, rank):
    from rlgpuschedule_b200 import synth
    return [synth.frame_gen(w['n_jobs'], w['seed0'] + rank * w['n_traces'] + i, w['n_jobs']) for i in range(w['n_traces'])]


def algorithmic_bytes(w, summ, n_nodes, n_gpus):
    """SURVEY.md 8(d), per replica-run.  fifo: 8Q + 12R + 12N + 8D + 64 per tick; sjf: 28 + 16 B per runnable job per event
    + 12N per event; dlas-gpu: 40 + 8 B per runnable job per event (sum_queued carries the swept runnable jobs there)."""
    if w['schedule'] == 'fifo':
        return 8 * summ['sum_queued'] + 12 * summ['sum_running'] + summ['n_ticks'] * (12 * n_nodes + 8 * n_gpus + 64)
    if w['schedule'] == 'sjf':
        return 44 * summ['sum_queued'] + 12 * n_nodes * summ['n_ticks']
    return 48 * summ['sum_queued']


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag, self.proc = index, [], False, None

    def run(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.samples.append([x.strip() for x in line.split(',')])
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc:
            try:
                self.proc.terminate()
            except Exception:
                pass
        sm = sorted(int(float(s[0])) for s in self.samples if s and s[0].replace('.', '').isdigit())
        mx = [int(float(s[1])) for s in self.samples if len(s) > 1 and s[1].replace('.', '').isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), s[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(self.samples))


# ------------------------------------------------------------------------------------------------ CPU side (oracle/ is touched only here)
def host_cores():
    """Threads this process may actually use (cgroup / affinity aware), not the machine's core count."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return os.cpu_count() or 1


def _cpu_sim():
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import cpu_sim
    cpu_sim.lib()
    return cpu_sim


def cpu_port_batch(cpu_sim, w, cl, traces, n_runs, threads):
    """n_runs replica-runs of the workload on `threads` host threads with the C port; returns events."""
    if w['schedule'] == 'fifo' and not w.get('env'):
        per = [n_runs // len(traces) + (1 if i < n_runs % len(traces) else 0) for i in range(len(traces))]
        return sum(cpu_sim.run_fifo_yarn_batch(cl, tr, n, threads, rows_cap=w['n_jobs'] + 16384) for tr, n in zip(traces, per) if n)
    from concurrent.futures import ThreadPoolExecutor   # ctypes releases the GIL inside the C call

    def one(i):
        tr = traces[i % len(traces)]
        if w.get('env'):
            o = cpu_sim.run_env_yarn(cl, tr, 1, window_k=5, seed=1, replica=i, rows_cap=w['n_jobs'] + 16384)
            return int((o['start'] >= 0).sum()) + int((o['end'] >= 0).sum()) + len(tr['nt'])
        o, _ = cpu_sim.run_legacy(cl, tr, w['schedule'], w['kw'].get('queue_limit', (30, 60, 150)))
        return o['counters']['events']
    with ThreadPoolExecutor(threads) as ex:
        return sum(ex.map(one, range(n_runs)))


def reference_python_sample(w):
    """The UNMODIFIED Python reference (staged by __graft_entry__.build() under oracle/_ref/reference) on this box's host:
    one process, one core, a 2 000-job trace of the same generator (the 60k-job trace takes 709 s, BASELINE.md).  fifo: the live
    simulator, `python run_sim.py`; sjf / dlas-gpu: the dead-code loops under the shim globals of oracle/ref_legacy_runner.py."""
    if not os.path.exists(os.path.join(REF_DIR, 'run_sim.py')) or w.get('env'):
        return None
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    os.environ['RLGS_REFERENCE_DIR'] = REF_DIR
    from rlgpuschedule_b200 import synth
    n = 2000
    work = tempfile.mkdtemp(prefix='rlgs_benchref_')
    fn = os.path.join(work, 'trace.csv')
    synth.write(synth.frame_gen(n, 1, n), fn)
    try:
        if w['schedule'] == 'fifo':
            import ref_runner
            ref_runner.REF = REF_DIR
            r = ref_runner.run_reference(fn, workdir=work, **CLUSTER_FLAGS)
            jobs = r['job_csv'].count('\r\n') - 1
            events = 3 * jobs
        else:
            import ref_legacy_runner
            ref_legacy_runner.REF = REF_DIR
            r = ref_legacy_runner.run_legacy(fn, w['schedule'], workdir=work, queue_limit=w['kw'].get('queue_limit', (30, 60, 150)), **CLUSTER_FLAGS)
            cpu_sim = _cpu_sim()
            o, _ = cpu_sim.run_legacy(cpu_sim.make_cluster(**CLUSTER_FLAGS), cpu_sim.prepare_trace(fn), w['schedule'], w['kw'].get('queue_limit', (30, 60, 150)))
            jobs, events = r['job_csv'].count('\r\n') - 1, o['counters']['events']   # the port equals these runs byte for byte: its event count is theirs
        return {'events_per_s': events / r['wall_s'], 'jobs_per_s': jobs / r['wall_s'], 'cores': 1, 'wall_s': round(r['wall_s'], 2),
                'sample': 'unmodified Python reference, %s, one process on one core, gen(%d, 1, %d) trace on the 4x32x8 cluster, wall time incl. interpreter start' % (
                    'python run_sim.py' if w['schedule'] == 'fifo' else 'dead-code loop under shim globals (oracle/ref_legacy_runner.py)', n, n)}
    except Exception as e:   # the baseline is a report, not a gate
        return {'error': str(e)[-300:]}


def cpu_baseline_sample(w):
    """Bounded cpu_baseline for the cuda arm's JSON line: a few seconds of the oracle port on every usable core."""
    cpu_sim = _cpu_sim()
    cores = host_cores()
    cl = cpu_sim.make_cluster(**CLUSTER_FLAGS)
    traces = [cpu_sim.prepare_trace(f) for f in frames(w, 0)[:2]]
    cpu_port_batch(cpu_sim, w, cl, traces, cores, cores)
    n_runs = (4 if w['n_jobs'] >= 60000 else 16) * cores
    t0 = time.perf_counter()
    ev = cpu_port_batch(cpu_sim, w, cl, traces, n_runs, cores)
    dt = time.perf_counter() - t0
    t1 = time.perf_counter()
    ev1 = cpu_port_batch(cpu_sim, w, cl, traces, 1, 1)
    dt1 = time.perf_counter() - t1
    out = {'value': ev / dt, 'unit': UNIT, 'cores': cores, 'kind': 'port',
           'sample': '%d replica-runs of the workload\'s trace on %d host threads, %.1f s (oracle/cpu_sim.c, gcc -O2)' % (n_runs, cores, dt),
           'single_core_value': ev1 / dt1}
    rp = reference_python_sample(w)
    if rp:
        out['reference_python'] = rp
    return out


def run_reference(args, w, rank):
    """CPU arm: the oracle port on all usable host cores, a bounded sample of the same workload per step."""
    if rank != 0:
        return
    cpu_sim = _cpu_sim()
    cores = host_cores()
    cl = cpu_sim.make_cluster(**CLUSTER_FLAGS)
    traces = [cpu_sim.prepare_trace(f) for f in frames(w, 0)[:min(w['n_traces'], 4)]]
    per_step = (2 if w['n_jobs'] >= 60000 else 8) * cores   # replica-runs per step

    def step():
        return cpu_port_batch(cpu_sim, w, cl, traces, per_step, cores)

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    ev = 0
    for _ in range(args.steps):
        ev += step()
    dt = time.perf_counter() - t0
    val = ev / dt
    sample = '%d replica-runs of the workload per step on %d host threads (oracle/cpu_sim.c, gcc -O2)' % (per_step, cores)
    cb = {'value': val, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': sample}
    rp = reference_python_sample(w) if not args.no_python_reference else None
    if rp:
        cb['reference_python'] = rp
    print(json.dumps({
        'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': 1e3 * dt / args.steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'int32', 'data': 'synthetic',
        'config': {'workload': '%s, %d replica-runs/step over %d seeds' % (w['text'], per_step, len(traces)), 'name': args.workload,
                   'note': 'CPU arm: bounded sample, host cores only; kind "port" = the C restatement pinned byte-for-byte on the reference\'s outputs'},
        'cpu_baseline': cb,
        'e2e': {'value': val, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }))


def bind_to_gpu_numa_node(index):
    """Pins this rank to the CPUs next to its GPU (NVML's ideal affinity) so that the pinned host mirrors it
    allocates are first-touched on the GPU's NUMA node: with several ranks per box the device->host copies
    otherwise cross the socket interconnect."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n_words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = {64 * w + b for w, word in enumerate(mask) for b in range(64) if (word >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
        return sorted(cpus)
    except Exception:
        return None


def load_profile(name):
    """profiles/r02_bench_profile.json: numbers read off the committed ncu captures of the CURRENT kernels (scripts/summarize_ncu.py)."""
    try:
        return json.load(open(os.path.join(ROOT, 'profiles', 'r02_bench_profile.json'))).get(name)
    except Exception:
        return None


def dump_outputs(out_dir, sim, env, R, rows, returns):
    """What the timed path returned in its last step, as float64 .npy files (at most 64 MB): `returns`, the episode return of
    every replica of every GPU (rank-major, as all-gathered); every summary field of this GPU's replicas; the job tables and, with
    rows, the per-tick / per-event rows of a seeded sample of this GPU's replicas (rows themselves a seeded sample above 65 536
    per replica; `rows_index` names them).  The arrays of the sampled replicas are concatenated in replica order; `<table>_len`
    holds each replica's length.  Rank 0 writes them."""
    import numpy as np
    from rlgpuschedule_b200 import _ffi
    rng = np.random.default_rng(0)
    out = {}

    def put(name, arrs):
        out[name] = np.concatenate([np.asarray(x, np.float64) for x in arrs])
        out[name + '_len'] = np.array([len(x) for x in arrs], np.float64)

    summ = [sim.summary(r) for r in range(R)]
    out.update({'summary_' + f: np.array([s[f] for s in summ], np.float64) for f, _ in _ffi.Summary._fields_})
    out['returns'] = np.asarray(returns, np.float64)
    if env is not None:
        out.update(env_obs=env.obs.double().cpu().numpy(), env_reward=env.reward.double().cpu().numpy(),
                   env_done=env.done.double().cpu().numpy())
    pick = np.sort(rng.choice(R, min(R, 4), replace=False))
    out['sample_replicas'] = pick.astype(np.float64)
    jobs = [sim.jobs(int(r)) for r in pick]
    for k in ('start', 'end', 'finish_order', 'preempt'):
        put('jobs_' + k, [j[k] for j in jobs])
    if rows:
        rs = [sim.rows(int(r)) for r in pick]
        idx = [np.sort(rng.choice(len(x), 65536, replace=False)) if len(x) > 65536 else np.arange(len(x)) for x in rs]
        put('rows_index', idx)
        for f in _ffi.ROW_DTYPE.names:
            out['rows_' + f] = np.concatenate([x[f][i].astype(np.float64) for x, i in zip(rs, idx)])
    bad = [name for name, a in out.items() if not np.isfinite(a).all()]
    assert not bad, 'outputs that are not finite: %s' % bad
    total = sum(a.nbytes for a in out.values())
    assert total <= 64 << 20, 'outputs to dump: %d bytes' % total
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='cuda', choices=['cuda', 'reference'])
    ap.add_argument('--workload', default='fifo60k', choices=sorted(WORKLOADS))
    ap.add_argument('--replicas', type=int, default=0, help='replicas per GPU (0 = the workload\'s default)')
    ap.add_argument('--lpr', type=int, default=0, help='fifo tick loop: lanes of a warp per replica (0 = chosen by the library)')
    ap.add_argument('--rows-format', default='event4', choices=['event4', 'event16', 'wire12', 'wire16', 'wide'])
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-python-reference', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write what the last timed step computed to DIR/<name>.npy (float64)')
    args = ap.parse_args()
    if args.dump_outputs and args.impl != 'cuda':
        ap.error('--dump-outputs writes what the timed cuda path computed: it needs --impl cuda')
    w = WORKLOADS[args.workload]
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if args.impl == 'reference':
        run_reference(args, w, rank)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import rlgpuschedule_b200 as rl
    from rlgpuschedule_b200 import _ffi
    if not torch.cuda.is_available():
        raise SystemExit('bench.py --impl cuda needs a CUDA device (no CPU fallback)')
    torch.cuda.set_device(local_rank)
    all_cpus = os.sched_getaffinity(0)
    bind_to_gpu_numa_node(local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    R = args.replicas or w['replicas']
    NT = w['n_traces']
    is_fifo = w['schedule'] == 'fifo'
    is_env = bool(w.get('env'))
    cluster = rl.Cluster(**CLUSTER_FLAGS)
    traces = [rl.prepare_trace(f, cluster) for f in frames(w, rank)]
    pinned = []   # the step's inputs (32-byte job records) live in pinned host memory: the e2e arm uploads them every step
    for tr in traces:
        try:
            buf = torch.from_numpy(np.ascontiguousarray(tr.records).view(np.uint8).copy()).pin_memory()
            tr.records = buf.numpy().view(_ffi.JOB_DTYPE)
            pinned.append(buf)
        except Exception as e:   # keeps the pageable arrays (slower uploads, same result)
            sys.stderr.write('bench: could not pin the trace records (%r)\n' % (e,))
            break
    bounds = [R * i // NT for i in range(NT + 1)]
    blocks = [(i, bounds[i], bounds[i + 1] - bounds[i]) for i in range(NT) if bounds[i + 1] > bounds[i]]
    sim_kw = dict(w['kw'])
    if is_fifo:
        sim_kw.update(lanes_per_replica=args.lpr, rows_format=args.rows_format)

    def attach(sim):
        for i, first, count in blocks:
            sim.load_trace(traces[i], first, count)

    class _Buf(object):
        def __init__(self, ptr, n):
            self.__cuda_array_interface__ = {'shape': (n,), 'typestr': '<i8', 'data': (ptr, False), 'version': 3}

    # ---------------- device-resident arm: `value`
    env = None
    if is_env:
        from rlgpuschedule_b200.env import Environment
        env = Environment(cluster, [(traces[i], first, count) for i, first, count in blocks], n_replicas=R, window_k=5, device=local_rank, seed=1)
        sim = env.sim
    else:
        sim = rl.Simulator(cluster, w['schedule'], w['scheme'], n_replicas=R, rows='device', device=local_rank, **sim_kw)
        attach(sim)
    ret_dev = torch.as_tensor(_Buf(sim.returns_device_ptr(), R), device='cuda') if world > 1 else None
    gathered = torch.empty(world * R, dtype=torch.int64, device='cuda') if world > 1 else None
    ev_k0, ev_k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    env_ms = [0.0]

    def step():
        if is_env:
            ev_k0.record()
            env.run_episodes('random')       # reset + device rollout of every episode + sync (regrows the slot table if a policy needs it)
            ev_k1.record()
            torch.cuda.synchronize()
            env_ms[0] = ev_k0.elapsed_time(ev_k1)
        else:
            sim.run()
        if world > 1:  # the one collective of the path: episode returns of every replica of every GPU
            dist.all_gather_into_tensor(gathered, ret_dev)

    for _ in range(max(args.warmup, 3)):
        step()
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    kernel_ms = 0.0
    launches = 0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
        if is_env:
            kernel_ms += env_ms[0]; launches += 2     # the zero-tick observation of reset() + the rollout
        else:
            ms, nl = sim.kernel_ms()
            kernel_ms += ms; launches += nl
    barrier()
    dt = time.perf_counter() - t0
    clocks = sampler.finish()
    summ = [sim.summary(first) for _, first, _ in blocks]
    cnt = [c for _, _, c in blocks]
    events_step = sum(s['events'] * c for s, c in zip(summ, cnt))
    jobs_step = sum(s['n_finished'] * c for s, c in zip(summ, cnt))
    ticks_step = sum(s['n_ticks'] * c for s, c in zip(summ, cnt))
    if is_env:   # every replica draws its own picks: count them all
        allsum = [sim.summary(r) for r in range(R)]
        events_step, jobs_step, ticks_step = (sum(s[k] for s in allsum) for k in ('events', 'n_finished', 'n_ticks'))
        summ, cnt = allsum, [1] * R
    alg_bytes_step = sum(algorithmic_bytes(w, s, cluster.num_nodes, cluster.num_gpus) * c for s, c in zip(summ, cnt))
    # job-updates (SURVEY 8d): queued + running jobs summed over the processed ticks (fifo) / runnable jobs swept per event (legacy)
    updates_step = sum((s['sum_queued'] + (s['sum_running'] if is_fifo else 0)) * c for s, c in zip(summ, cnt))
    lpr_used = None
    t = torch.tensor([dt, kernel_ms / 1e3], dtype=torch.float64, device='cuda')
    tot = torch.tensor([events_step, jobs_step, ticks_step, updates_step], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        if rank == 0:
            g = gathered.cpu().numpy().reshape(world, R)
            assert (g[0] == sim.returns()).all(), 'all-gathered returns do not match the local ones'
    dt_max, kern_s = t.tolist()
    events_all, jobs_all, ticks_all, updates_all = tot.tolist()
    value = events_all * args.steps / dt_max
    jmax = max(len(tr.records) for tr in traces)
    max_ticks = max(s['n_ticks'] for s in summ)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, sim, env, R, rows=not is_env, returns=gathered.cpu().numpy() if world > 1 else sim.returns())
    (env or sim).close()

    # ---------------- end-to-end arm through the C ABI with host buffers
    def e2e_arm(rows_format):
        """Every step: records host -> device, simulate, the result of every replica device -> pinned host memory."""
        if is_env:
            env2 = Environment(cluster, [(traces[i], first, count) for i, first, count in blocks], n_replicas=R, window_k=5, device=local_rank, seed=1)

            def step2():
                for i, first, count in blocks:            # host -> device: the episode's traces
                    env2.sim.load_trace(traces[i], first, count)
                env2.run_episodes('random')
                return env2.sim.returns()                  # device -> host: episode returns
            closer = env2
        else:
            kw2 = dict(sim_kw)
            if is_fifo:
                kw2['rows_format'] = rows_format
            sim2 = rl.Simulator(cluster, w['schedule'], w['scheme'], n_replicas=R, rows='host', fetch_jobs=(False if rows_format.startswith('event') else 'end') if is_fifo else True, device=local_rank, **kw2)
            attach(sim2)

            def step2():
                attach(sim2)          # host -> device: the step's input records
                sim2.run()            # simulate; rows (+ job tables, format permitting) -> pinned host store, overlapped with compute
                return int(sim2.summary(0)['n_finished'])
            closer = sim2
        for _ in range(max(args.warmup, 3)):
            step2()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step2()
        barrier()
        dt2 = time.perf_counter() - t0
        t2 = torch.tensor([dt2], dtype=torch.float64, device='cuda')
        if world > 1:
            dist.all_reduce(t2, op=dist.ReduceOp.MAX)
        h2d = sum(len(traces[i].records) * 32 for i, _, _ in blocks)
        if is_env:
            d2h = 8 * R + R * 264
        else:
            rows0 = sim2.rows(0)
            j0 = sim2.jobs(0)
            assert len(rows0) == summ[0]['n_ticks'] and int(rows0['finished'][-1]) == len(j0['finish_order'])
            row_bytes = {'event4': 4, 'event16': 16, 'wire12': 12, 'wire16': 16, 'wide': 64}[rows_format] if is_fifo else 64
            n_planes = (0 if rows_format.startswith('event') else 2) if is_fifo else 3
            n_chunks = -(-max_ticks // _ffi.ROWS_PER_CHUNK)        # whole chunks travel (chunk-major row store)
            d2h = int(n_chunks * R * _ffi.ROWS_PER_CHUNK * row_bytes + n_planes * 4 * R * jmax + R * 264)   # rows + job tables + replica states
        out = {'value': events_all * args.steps / t2.item(), 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
               'ms_per_step': 1e3 * t2.item() / args.steps}
        closer.close()
        return out

    e2e = e2e_stat_rows = None
    if not args.no_e2e:
        e2e = e2e_arm(args.rows_format)
        if is_fifo and not is_env and args.rows_format == 'event4':
            # companion number: the same step with the rows that still carry the kernel-computed pending-time statistics
            e2e_stat_rows = e2e_arm('event16')
            e2e_stat_rows['rows_format'] = 'event16'
            e2e_stat_rows['note'] = ('16 bytes per tick: max / median pending times computed by the kernel + the job started at the tick; the default '
                                     '(event4) sends the event log alone and the library derives those columns on the host when a replica is read')

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except Exception:
            pass
        hbm_peak = float(peaks.get('hbm_gbs', 6650.0))
        per_launch_s = kern_s / args.steps
        alg_gbps = alg_bytes_step / per_launch_s / 1e9
        prof = load_profile(args.workload) or {}
        kernel_name = {'fifo': 'fifo_grp_kernel', 'sjf': 'sjf_yarn_kernel', 'dlas-gpu': 'dlas_gpu_kernel'}[w['schedule']]
        # bytes per replica-tick (fifo) / per swept job (legacy) that the committed ncu capture of this kernel measured in DRAM
        traffic = None
        if prof.get('dram_bytes_per_unit') is not None:
            units = ticks_step if is_fifo else sum(s['sum_queued'] * c for s, c in zip(summ, cnt))
            traffic = prof['dram_bytes_per_unit'] * units
        if is_fifo:
            # the tick loop keeps the state SURVEY 8(d) counts in shared memory / registers: it is bound by instruction issue.
            # achieved = warp instructions per replica-tick (ncu capture of THIS kernel) x replica-ticks/s measured now
            sm_hz = 1e6 * float(clocks.get('sm_mhz') or 1965)
            peak_issue = 148 * 4 * sm_hz / 1e9
            ipt = prof.get('warp_inst_per_replica_tick')
            ach = ipt * (ticks_step / per_launch_s) / 1e9 if ipt else None
            roofline = {'bound': 'issue', 'achieved': ach, 'peak': peak_issue, 'unit': 'Gwarp-inst/s', 'frac': (ach / peak_issue) if ach else None,
                        'traffic': traffic, 'warp_inst_per_replica_tick': ipt,
                        'peak_source': '148 SMs x 4 schedulers x 1 warp-inst/clk at the SM clock sampled during the run',
                        'profile': prof.get('source'),
                        'algorithmic_equiv_GBps': alg_gbps, 'hbm_peak_GBps': hbm_peak,
                        'dram_GBps': (traffic / per_launch_s / 1e9) if traffic else None,
                        'dram_frac': (traffic / per_launch_s / 1e9 / hbm_peak) if traffic else None,
                        'note': 'the per-tick state SURVEY 8(d) counts (8Q+12R+12N+8D+64 B) lives on chip, so algorithmic_equiv_GBps is not a bandwidth '
                                'the kernel must sustain; ncu shows instruction issue as the limiter and DRAM at a few % of peak'}
        else:
            roofline = {'bound': 'hbm', 'achieved': alg_gbps, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': alg_gbps / hbm_peak, 'traffic': traffic,
                        'peak_source': 'MEASURED_PEAKS.json hbm_gbs' if 'hbm_gbs' in peaks else 'fallback 6650 GB/s',
                        'profile': prof.get('source'),
                        'dram_GBps': (traffic / per_launch_s / 1e9) if traffic else None,
                        'dram_frac': (traffic / per_launch_s / 1e9 / hbm_peak) if traffic else None,
                        'issue_active_pct_in_profile': prof.get('issue_active_pct'),
                        'note': 'achieved = SURVEY 8(d) algorithmic bytes of the per-event sweep (runnable entries streamed 32 at a time) / kernel time; '
                                'the entry lists mostly live in L2, and the ncu capture shows the kernel closer to the issue limit than to the DRAM one'}
        roofline['launch'] = 'one step = %d launches of %s; bytes and time are per step' % (launches // max(args.steps, 1), kernel_name)
        out = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
            'ms_per_step': 1e3 * dt_max / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'int32', 'data': 'synthetic',
            'config': {'workload': '%s, %d replicas/GPU over %d seeds' % (w['text'], R, NT), 'name': args.workload, 'schedule': w['schedule'],
                       'scheme': w['scheme'], 'replicas_per_gpu': R, 'jobs_per_replica': w['n_jobs'],
                       'rows_format': (args.rows_format if is_fifo and not is_env else ('none' if is_env else 'wide')),
                       'e2e_result': (('4-byte event rows (idle nodes | the queue head started | queue length): the event log of every replica; rlgs_read_jobs / '
                                       'rlgs_read_rows replay the queue on the host to rebuild start / end / finish-order and the per-tick statistics of a replica '
                                       'when asked for (tests compare them with the device-written tables and the 64-byte rows); --rows-format wide|wire16|wire12|event16 '
                                       'move progressively fewer derived bytes' if args.rows_format == 'event4' else
                                       '16-byte event rows: the per-tick statistics + the job started at the tick; start / end / finish-order tables are rebuilt from '
                                       'them on the host when asked for (end = start + dur_ticks, finish order = (end, start))' if args.rows_format == 'event16' else
                                       'per-tick rows in the wire format + end_tick and finish_order per job (fifo: start = end - dur_ticks, derived on the host)')
                                      if is_fifo and not is_env else ('episode returns' if is_env else 'per-event rows + start / end / finish_order per job')),
                       'lanes_per_replica': (args.lpr or 'auto') if is_fifo else 32,
                       'replica_note': 'replicas of one seed compute identical deterministic simulations (fifo / sjf / dlas draw nothing); the kernel '
                                       'puts replicas a quarter of a launch apart into one warp, so the replicas sharing a warp follow different seeds',
                       'l2': 'per-step working set (queue stacks + row store + job tables) >> 126 MB L2; no explicit flush',
                       'parallelism': 'replicas: %d GPU x %d (share-nothing), one all-gather of returns' % (world, R)},
            'jobs_per_sec': jobs_all * args.steps / dt_max, 'ticks_per_sec': ticks_all * args.steps / dt_max,
            'job_updates_per_sec': updates_all * args.steps / dt_max,
            'gpu_launches': launches, 'kernel_ms_per_step': 1e3 * per_launch_s,
            'roofline': roofline, 'clocks': clocks,
        }
        if e2e:
            out['e2e'] = e2e
        if e2e_stat_rows:
            out['e2e_stat_rows'] = e2e_stat_rows
        if not args.no_cpu and world == 1:   # the CPU baseline is reported at N=1 only, on every usable host core
            os.sched_setaffinity(0, all_cpus)
            out['cpu_baseline'] = cpu_baseline_sample(w)
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
