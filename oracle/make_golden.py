"""Generate tests/golden/* by running the real reference (oracle/ref_runner.py) in this container.

    python oracle/make_golden.py [case ...]        # default: every case not yet generated
    python oracle/make_golden.py --random          # the random cases of golden_cases.RANDOM_* -> tests/golden/random_cases.json.gz

Per case it stores: trace.csv (small cases; big ones are regenerated from tracegen seeds and
checked by sha256), job.csv and cluster_noutil.csv exactly as the reference wrote them (CRLF
line ends; gzip for big cases), and meta.json (flags, hashes, tick count, reference wall time).
`cluster_noutil` = cluster.csv without the avg_gpu_utilization column (unseeded RNG in the
reference, /root/reference/infra/device.py:52).
"""
import gzip
import hashlib
import json
import os
import sys
import tempfile
from concurrent.futures import ProcessPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import golden_cases  # noqa: E402
import ref_runner  # noqa: E402
import tracegen  # noqa: E402

ROOT = os.path.dirname(HERE)
GOLD = os.path.join(ROOT, 'tests', 'golden')


def sha(b):
    if isinstance(b, str):
        b = b.encode()
    return hashlib.sha256(b).hexdigest()


def make(name):
    case = golden_cases.CASES[name]
    out = os.path.join(GOLD, name)
    os.makedirs(out, exist_ok=True)
    big = case.get('big', False)
    work = tempfile.mkdtemp(prefix='rlgs_gold_%s_' % name)
    trace = os.path.join(work, 'trace.csv')
    tracegen.write(case['frame'](), trace)
    flags = dict(case['flags'])
    for k, v in list(flags.items()):
        if isinstance(v, str) and v.startswith('@'):
            flags[k] = os.path.join(ROOT, v[1:])
    sched = case.get('schedule', 'fifo')
    if sched in golden_cases.LEGACY:
        return make_legacy(name, case, out, work, trace, flags, big)
    if sched != 'fifo':   # the pack placements are keyed by the schedule name (schedule.py:47)
        flags.update(schedule=sched, scheme=case.get('scheme', sched), num_buffer=case.get('num_buffer', 5))
    if sched == 'horus+':   # k-means queues: the draws of np.random.randint / choice are injected (ref_runner._INJECT)
        flags.update(num_queue=case['num_queue'], inject_seed=case['inject_seed'])
    res = ref_runner.run_reference(trace, workdir=work, **flags)
    job, clu = res['job_csv'], res['cluster_csv']
    if job is None or clu is None:
        raise RuntimeError('%s: reference failed: %s' % (name, res['stderr']))
    noutil = ref_runner.strip_util_column(clu)
    trace_bytes = open(trace, 'rb').read()
    meta = dict(case=name, flags=case['flags'], schedule=sched, scheme=case.get('scheme', sched if sched != 'fifo' else 'yarn'), num_buffer=case.get('num_buffer', 5), num_queue=case.get('num_queue', 1), inject_seed=case.get('inject_seed'), trace_sha256=sha(trace_bytes),
                job_sha256=sha(job), cluster_noutil_sha256=sha(noutil),
                n_job_rows=job.count('\r\n') - 1, n_ticks=clu.count('\r\n') - 1,
                reference_wall_s=round(res['wall_s'], 2), reference_returncode=res['returncode'],
                generated_with='python %s numpy/pandas as in this image; reference @ /root/reference' % sys.version.split()[0])
    if not big:
        open(os.path.join(out, 'trace.csv'), 'wb').write(trace_bytes)
        open(os.path.join(out, 'job.csv'), 'w', newline='').write(job)
        open(os.path.join(out, 'cluster_noutil.csv'), 'w', newline='').write(noutil)
    elif not case.get('huge', False):
        with gzip.GzipFile(os.path.join(out, 'job.csv.gz'), 'wb', mtime=0) as f:
            f.write(job.encode())
        with gzip.GzipFile(os.path.join(out, 'cluster_noutil.csv.gz'), 'wb', mtime=0) as f:
            f.write(noutil.encode())
    json.dump(meta, open(os.path.join(out, 'meta.json'), 'w'), indent=1, sort_keys=True)
    return name, meta['n_ticks'], meta['n_job_rows'], meta['reference_wall_s']


def make_legacy(name, case, out, work, trace, flags, big):
    """sjf / shortest / shortest-gpu / dlas-gpu / dlas: the reference's dead-code loops run unmodified under shim globals
    (oracle/ref_legacy_runner.py); job.csv and cluster.csv are the files the reference's own log._Log wrote."""
    import ref_legacy_runner
    sched = case['schedule']
    ql = tuple(case.get('queue_limit', ()))
    res = ref_legacy_runner.run_legacy(trace, sched, workdir=work, queue_limit=ql or (30, 60, 150), **flags)
    job, clu = res['job_csv'], res['cluster_csv']
    trace_bytes = open(trace, 'rb').read()
    meta = dict(case=name, flags=case['flags'], schedule=sched, scheme='count' if sched in ('dlas-gpu', 'dlas') else 'yarn', queue_limit=list(ql),
                trace_sha256=sha(trace_bytes), job_sha256=sha(job), cluster_sha256=sha(clu), n_job_rows=job.count('\r\n') - 1,
                n_events=clu.count('\r\n') - 1, reference_wall_s=round(res['wall_s'], 2),
                generated_with='python %s; reference dead code run_sim.py run unmodified by oracle/ref_legacy_runner.py (shim JOBS / scheduler)' % sys.version.split()[0])
    if not big:
        open(os.path.join(out, 'trace.csv'), 'wb').write(trace_bytes)
        open(os.path.join(out, 'job.csv'), 'w', newline='').write(job)
        open(os.path.join(out, 'cluster.csv'), 'w', newline='').write(clu)
    elif not case.get('huge', False):
        with gzip.GzipFile(os.path.join(out, 'job.csv.gz'), 'wb', mtime=0) as f:
            f.write(job.encode())
        with gzip.GzipFile(os.path.join(out, 'cluster.csv.gz'), 'wb', mtime=0) as f:
            f.write(clu.encode())
    json.dump(meta, open(os.path.join(out, 'meta.json'), 'w'), indent=1, sort_keys=True)
    return name, meta['n_events'], meta['n_job_rows'], meta['reference_wall_s']


def _random_one(arg):
    """One random case through the reference: its files, the sha256 of the trace it read, and how it ended."""
    family, seed, rest = arg
    work = tempfile.mkdtemp(prefix='rlgs_gold_random_%d_' % seed)
    trace = os.path.join(work, 't.csv')
    if family == 'legacy':
        import ref_legacy_runner
        df, flags = golden_cases.random_case(seed)
        tracegen.write(df, trace)
        ql = golden_cases.random_legacy_queue_limit(seed)
        res = ref_legacy_runner.run_legacy(trace, rest[0], workdir=work, queue_limit=ql, **flags)
        clu = res['cluster_csv']
    else:
        if family == 'fifo':
            df, flags = golden_cases.random_case(seed)
            extra = {}
        else:
            sched, scheme = rest
            df, flags, k, kq, inj = golden_cases.random_pack_case(seed, sched, scheme)
            extra = dict(schedule=sched, scheme=scheme, num_buffer=k, **(dict(num_queue=kq, inject_seed=inj) if sched == 'horus+' else {}))
        tracegen.write(df, trace)
        res = ref_runner.run_reference(trace, workdir=work, **extra, **flags)
        clu = ref_runner.strip_util_column(res['cluster_csv']) if res['cluster_csv'] is not None else None
    rec = dict(trace_sha256=sha(open(trace, 'rb').read()), job_csv=res['job_csv'], cluster_csv=clu,
               returncode=res.get('returncode'), stderr_has_error='Error' in res['stderr'])
    return golden_cases.random_key(family, seed, *rest), rec


def make_random():
    args = ([('fifo', s, ()) for s in golden_cases.RANDOM_FIFO] + [('pack', s, combo) for s, combo in golden_cases.RANDOM_PACK]
            + [('legacy', s, (sched,)) for s, sched in golden_cases.RANDOM_LEGACY])
    with ProcessPoolExecutor(max_workers=int(os.environ.get('GOLD_JOBS', '6'))) as ex:
        out = dict(ex.map(_random_one, args))
    fn = os.path.join(GOLD, golden_cases.RANDOM_GOLD)
    with gzip.GzipFile(fn, 'wb', mtime=0) as f:
        f.write(json.dumps(out, indent=0, sort_keys=True).encode())
    return fn, len(out)


if __name__ == '__main__':
    if sys.argv[1:] == ['--random']:
        print(*make_random())
        sys.exit(0)
    names = sys.argv[1:] or [n for n in golden_cases.CASES
                             if not os.path.exists(os.path.join(GOLD, n, 'meta.json'))]
    with ProcessPoolExecutor(max_workers=int(os.environ.get('GOLD_JOBS', '6'))) as ex:
        for r in ex.map(make, names):
            print(*r, flush=True)
