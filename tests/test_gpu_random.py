"""Randomised differential tests on the device: 60 random traces x cluster shapes, every schedule, against the
CPU oracle (which tests/test_oracle_vs_live_reference.py ties to the reference's recorded files on the same generator)."""
import numpy as np
import pytest

import cpu_sim
from golden_cases import random_case
import rlgpuschedule_b200 as rl
from rlgpuschedule_b200 import _ffi, log_manager as lm, synth

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize('block', range(6))
def test_random_cases_all_schedules(block):
    for seed in range(200 + 10 * block, 210 + 10 * block):
        df, flags = random_case(seed)
        cluster = rl.cluster_from_flags(flags)
        tr = rl.prepare_trace(df, cluster)
        otr = cpu_sim.prepare_trace(df)
        oc = cpu_sim.make_cluster(**flags)
        # fifo: CSV text must match the oracle's
        sim = rl.Simulator(cluster, 'fifo', 'yarn', n_replicas=2, rows=True, ticks_per_launch=int(3 + seed % 11))
        sim.load_trace(tr); sim.run()
        o = cpu_sim.run_fifo_yarn(oc, otr)
        j = sim.jobs(1)
        assert lm.format_job_csv(tr, j['finish_order'], j['start'], j['end'], j['preempt']) == cpu_sim.format_job_csv(otr, o), seed
        assert lm.format_cluster_csv(sim.rows(1), cluster, tr.mem_shift, with_util=False) == cpu_sim.format_cluster_csv(o), seed
        sim.close()
        for sched, scheme, kw, run in (('sjf', 'yarn', {}, lambda: cpu_sim.run_sjf_yarn(oc, otr)),
                                       ('shortest', 'yarn', {}, lambda: cpu_sim.run_sjf_yarn(oc, otr, sort_mode=1)),
                                       ('shortest-gpu', 'yarn', {}, lambda: cpu_sim.run_sjf_yarn(oc, otr, sort_mode=2)),
                                       ('dlas', 'count', dict(num_queue=3, queue_limit=(3, 11)), lambda: cpu_sim.run_dlas_gpu(oc, otr, (3, 11), gputime=False)),
                                       ('dlas-gpu', 'count', dict(num_queue=3, queue_limit=(6, 40)), lambda: cpu_sim.run_dlas_gpu(oc, otr, (6, 40)))):
            sim = rl.Simulator(cluster, sched, scheme, n_replicas=1, rows=True, **kw)
            sim.load_trace(tr); sim.run()
            o = run()
            j = sim.jobs(0)
            for k in ('finish_order', 'start', 'end', 'preempt'):
                assert np.array_equal(j[k], o[k]), (seed, sched, k)
            assert np.array_equal(sim.job_plane(0, _ffi.PLANE_AUX), o['pending']), (seed, sched)
            rows = sim.rows(0)
            assert np.array_equal(rows['median_lo'], o['rows']['time']) and np.array_equal(rows['busy_gpus'], o['rows']['busy_gpus']), (seed, sched)
            assert np.array_equal(rows['idle_nodes'], o['rows']['idle_nodes']) and np.array_equal(rows['queued'], o['rows']['pending']), (seed, sched)
            sim.close()


PACK_COMBOS = [('horus', 'horus'), ('gandiva', 'gandiva'), ('horus+', 'horus+'), ('horus', 'yarn'), ('gandiva', 'yarn'), ('horus+', 'yarn')]


@pytest.mark.parametrize('sched,scheme', PACK_COMBOS)
def test_random_cases_pack_family(sched, scheme):
    """The same generator as the oracle's differential test against the reference (tests/test_oracle_vs_live_reference.py): device vs oracle
    on random traces / cluster shapes / look-ahead / queue counts, mean and seeded utilisation draws."""
    for seed in range(300, 312):
        df, flags = random_case(seed)
        rng = np.random.default_rng(seed + 7)
        k = int(rng.integers(1, 8)); kq = int(rng.integers(1, 5)); inj = int(rng.integers(1, 1000))
        draws = bool(seed % 3 == 0) and scheme != 'yarn'        # every third case: seeded utilisation draws on the real spread
        if scheme != 'yarn' and not draws:
            df = df.copy(); df['gpu_utilization_max'] = df['gpu_utilization_avg']
        cluster = rl.cluster_from_flags(flags)
        tr = rl.prepare_trace(df, cluster)
        otr = cpu_sim.prepare_trace(df)
        try:
            o = cpu_sim.run_pack(cpu_sim.make_cluster(**flags), otr, sched, k, scheme=('yarn' if scheme == 'yarn' else None),
                                 num_queue=kq, inject_seed=inj, seed=(inj if draws else None), replica=1)
        except RuntimeError:
            continue                                             # the reference would raise on this input
        kw = dict(num_queue=kq) if sched == 'horus+' else {}
        sim = rl.Simulator(cluster, sched, scheme, n_replicas=2, rows=True, num_buffer=k, pack_seed=inj, pack_rng=draws,
                           max_ticks=400000, ticks_per_launch=int(seed % 4) * 29, **kw)
        sim.load_trace(tr); sim.run()
        j = sim.jobs(1)
        dur = tr.duration + 5.0 * (sim.job_plane(1, _ffi.PLANE_AUX) == 1)
        job = lm.format_job_csv(tr, j['finish_order'], j['start'], j['end'], j['preempt'], get_duration=dur, jct=sim.job_plane(1, _ffi.PLANE_PREEMPT))
        assert job == cpu_sim.format_job_csv(otr, o), (seed, sched, scheme)
        assert lm.format_cluster_csv(sim.rows(1), cluster, tr.mem_shift, with_util=False) == cpu_sim.format_cluster_csv(o), (seed, sched, scheme)
        sim.close()
