"""Registry of parity cases shared by oracle/make_golden.py (which runs the real reference in
this container) and tests/ (which replay the same traces through oracle/cpu_sim.c and the CUDA
path).  Test infrastructure only.

Each case: name -> dict(frame=callable returning the trace DataFrame, flags=dict of run_sim.py
cluster flags, big=bool (fixture stored gzip'ed / hashed instead of plain text)).
Edge cases follow the quirk list in SURVEY.md Appendix A (q1..q13).
"""
import numpy as np

import tracegen as tg

C148 = dict(num_switch=1, num_node_p_switch=4, num_gpu_p_node=8)
C4328 = dict(num_switch=4, num_node_p_switch=32, num_gpu_p_node=8)


def _kat6(drop_last=False):
    rows = [dict(normalized_time=0, minutes=20, used_gpus=8.0, gpu_per_container=8),
            dict(normalized_time=10000, minutes=4, used_gpus=8.0, gpu_per_container=8),
            dict(normalized_time=20000, minutes=4, used_gpus=8.0, gpu_per_container=8),
            dict(normalized_time=30000, minutes=4, used_gpus=4.0, gpu_per_container=4),
            dict(normalized_time=30000, minutes=4, used_gpus=4.0, gpu_per_container=4),
            dict(normalized_time=600000, minutes=2, used_gpus=1.0, gpu_per_container=1)]
    if drop_last:
        rows = rows[:-1]
    return tg.frame_rows(rows)


def _multi_node():
    # 2 switches x 2 nodes x 4 GPUs: cross-node yarn (gpus > 4), the `<=` off-by-one (q11),
    # least_num_full_nodes, and a job that can never be placed (9 GPUs in one 8-GPU task).
    rows = [dict(normalized_time=0, minutes=30, used_gpus=8.0, gpu_per_container=4),
            dict(normalized_time=11000, minutes=12, used_gpus=6.0, gpu_per_container=2),
            dict(normalized_time=23000, minutes=8, used_gpus=5.0, gpu_per_container=1),
            dict(normalized_time=31000, minutes=9, used_gpus=2.0, gpu_per_container=1),
            dict(normalized_time=45000, minutes=20, used_gpus=16.0, gpu_per_container=2),
            dict(normalized_time=52000, minutes=5, used_gpus=3.0, gpu_per_container=3),
            dict(normalized_time=90000, minutes=7, used_gpus=12.0, gpu_per_container=4),
            dict(normalized_time=150000, minutes=3, used_gpus=4.0, gpu_per_container=4),
            dict(normalized_time=400000, minutes=6, used_gpus=1.0, gpu_per_container=1),
            dict(normalized_time=410000, minutes=6, used_gpus=9.0, gpu_per_container=8),
            dict(normalized_time=900000, minutes=2, used_gpus=1.0, gpu_per_container=1)]
    return tg.frame_rows(rows)


def _resource_bound(seed):
    rng = np.random.default_rng(seed)
    n = 60
    g = rng.choice([1, 2, 4, 8, 16], n, p=[.4, .2, .2, .15, .05])
    gpc = np.minimum(g, rng.choice([1, 2, 4], n))
    gpc = np.where(g % gpc == 0, gpc, 1)
    rows = [dict(normalized_time=float(t), minutes=float(m), used_gpus=float(a), gpu_per_container=int(b))
            for t, m, a, b in zip(np.sort(rng.uniform(0, 3e6, n)), rng.uniform(2, 80, n), g, gpc)]
    return tg.frame_rows(rows)


def _big_mem():
    # memory_max above cap-500 MiB: no device accepts the task and the reference leaks
    # cpu_used/mem_used on every visited node every tick (q8).  Newer arrivals jump the queue (q1).
    rows = [dict(normalized_time=0, minutes=10, used_gpus=2.0, gpu_per_container=1),
            dict(normalized_time=20000, minutes=6, used_gpus=2.0, gpu_per_container=1, memory_max=40000000000),
            dict(normalized_time=50000, minutes=6, used_gpus=1.0, gpu_per_container=1),
            dict(normalized_time=90000, minutes=4, used_gpus=12.0, gpu_per_container=4, memory_max=36000000000),
            dict(normalized_time=120000, minutes=8, used_gpus=4.0, gpu_per_container=2),
            dict(normalized_time=300000, minutes=3, used_gpus=8.0, gpu_per_container=8),
            dict(normalized_time=700000, minutes=2, used_gpus=1.0, gpu_per_container=1)]
    return tg.frame_rows(rows)


def _nondivisible():
    rows = [dict(normalized_time=0, minutes=9, used_gpus=3.0, gpu_per_container=2),
            dict(normalized_time=10000, minutes=7, used_gpus=6.0, gpu_per_container=4),
            dict(normalized_time=12000, minutes=11, used_gpus=12.0, gpu_per_container=5),
            dict(normalized_time=30000, minutes=5, used_gpus=7.0, gpu_per_container=2),
            dict(normalized_time=35000, minutes=3, used_gpus=8.0, gpu_per_container=3),
            dict(normalized_time=250000, minutes=2, used_gpus=1.0, gpu_per_container=1)]
    return tg.frame_rows(rows)


def _filter_nan():
    # q13: interactive rows and rows with NaN are dropped; input unsorted; first arrival != 0.
    rows = [dict(normalized_time=530000, minutes=6, used_gpus=2.0, gpu_per_container=2),
            dict(normalized_time=500000, minutes=3, used_gpus=1.0, gpu_per_container=1, type='interactive'),
            dict(normalized_time=512345, minutes=14.5, used_gpus=8.0, gpu_per_container=4),
            dict(normalized_time=505000, minutes=np.nan, used_gpus=1.0, gpu_per_container=1),
            dict(normalized_time=641000, minutes=2.2, used_gpus=4.0, gpu_per_container=1),
            dict(normalized_time=511111, minutes=1.0, used_gpus=1.0, gpu_per_container=1),
            dict(normalized_time=700000, minutes=5, used_gpus=1.0, gpu_per_container=1, memory_avg=np.nan),
            dict(normalized_time=909090, minutes=0.9, used_gpus=1.0, gpu_per_container=1)]
    return tg.frame_rows(rows)


def _short():
    # cf5: runtime = max(1, ceil(minutes*0.5)); includes duration 0, 0.25, exactly 1.0 and 2.0
    mins = [0.0, 0.5, 2.0, 4.0, 4.0000001, 1.999999, 3.0, 0.01, 6.0, 2.0]
    rows = [dict(normalized_time=7000.0 * i, minutes=m, used_gpus=2.0, gpu_per_container=2)
            for i, m in enumerate(mins)]
    return tg.frame_rows(rows)


def _ties():
    # batches of simultaneous arrivals (front insertion keeps batch order, q1) under load
    rng = np.random.default_rng(11)
    rows = []
    for b in range(12):
        t = float(b * 40000 + 5000)
        for _ in range(int(rng.integers(1, 6))):
            g = int(rng.choice([1, 2, 4, 8]))
            rows.append(dict(normalized_time=t, minutes=float(rng.uniform(3, 40)), used_gpus=float(g),
                             gpu_per_container=int(rng.choice([1, g]))))
    rows.append(dict(normalized_time=2.5e6, minutes=2, used_gpus=1.0, gpu_per_container=1))
    return tg.frame_rows(rows)


def _zs(frame):
    """Zero utilisation spread: gpu_utilization_max = gpu_utilization_avg makes every np.random.normal(loc, 0) of
    infra/device.py:30,52 return loc, so the reference's horus path is deterministic and can be pinned."""
    def f():
        df = frame().copy()
        df['gpu_utilization_max'] = df['gpu_utilization_avg']
        return df
    return f


CASES = {
    'kat6': dict(frame=_kat6, flags=dict(num_switch=1, num_node_p_switch=1, num_gpu_p_node=8)),
    'kat5_early': dict(frame=lambda: _kat6(True), flags=dict(num_switch=1, num_node_p_switch=1, num_gpu_p_node=8)),
    'probe100': dict(frame=tg.frame_probe100, flags=C148),
    'multi_node': dict(frame=_multi_node, flags=dict(num_switch=2, num_node_p_switch=2, num_gpu_p_node=4)),
    'cpu_bound': dict(frame=lambda: _resource_bound(21), flags=dict(num_switch=1, num_node_p_switch=6, num_gpu_p_node=8, num_cpu_p_node=30)),
    'mem_bound': dict(frame=lambda: _resource_bound(22), flags=dict(num_switch=2, num_node_p_switch=3, num_gpu_p_node=8, mem_p_node=130)),
    'big_mem_leak': dict(frame=_big_mem, flags=dict(num_switch=1, num_node_p_switch=3, num_gpu_p_node=4, num_cpu_p_node=64, mem_p_node=256)),
    'gpu_cap16': dict(frame=lambda: tg.frame_gen(120, 7, 150), flags=dict(num_switch=1, num_node_p_switch=8, num_gpu_p_node=8, gpu_memory_capacity=12)),
    'nondivisible': dict(frame=_nondivisible, flags=dict(num_switch=1, num_node_p_switch=2, num_gpu_p_node=8)),
    'filter_nan': dict(frame=_filter_nan, flags=C148),
    'short_durations': dict(frame=_short, flags=dict(num_switch=1, num_node_p_switch=1, num_gpu_p_node=4)),
    'ties': dict(frame=_ties, flags=dict(num_switch=1, num_node_p_switch=2, num_gpu_p_node=8)),
    'cluster_spec': dict(frame=lambda: tg.frame_gen(150, 9, 400), flags=dict(cluster_spec='@examples/cluster_spec_2x8x4.csv')),
    'dense': dict(frame=lambda: tg.frame_gen(300, 5, 30), flags=dict(num_switch=2, num_node_p_switch=4, num_gpu_p_node=8)),
    'probe2k': dict(frame=lambda: tg.frame_gen(2000, 1, 2000), flags=C4328, big=True),
    'probe10k': dict(frame=lambda: tg.frame_gen(10000, 2, 10000), flags=C4328, big=True),
    'loaded10k': dict(frame=lambda: tg.frame_gen(10000, 4, 2500), flags=C4328, big=True),
    'probe60k': dict(frame=lambda: tg.frame_gen(60000, 3, 60000), flags=C4328, big=True, huge=True),
    # --schedule horus --scheme horus (schedule_horus + horus_placement), zero-spread traces
    'horus_probe100': dict(frame=_zs(tg.frame_probe100), flags=C148, schedule='horus'),
    'horus_racks_k3': dict(frame=_zs(tg.frame_probe100), flags=dict(num_switch=2, num_node_p_switch=2, num_gpu_p_node=8), schedule='horus', num_buffer=3),
    'horus_multi_node': dict(frame=_zs(_multi_node), flags=dict(num_switch=2, num_node_p_switch=2, num_gpu_p_node=4), schedule='horus'),
    'horus_big_mem_leak': dict(frame=_zs(_big_mem), flags=dict(num_switch=1, num_node_p_switch=3, num_gpu_p_node=4, num_cpu_p_node=64, mem_p_node=256), schedule='horus'),
    'horus_gpu_cap16': dict(frame=_zs(lambda: tg.frame_gen(120, 7, 150)), flags=dict(num_switch=1, num_node_p_switch=8, num_gpu_p_node=8, gpu_memory_capacity=12), schedule='horus'),
    'horus_ties': dict(frame=_zs(_ties), flags=dict(num_switch=1, num_node_p_switch=2, num_gpu_p_node=8), schedule='horus'),
    'horus_mem_bound': dict(frame=_zs(lambda: _resource_bound(22)), flags=dict(num_switch=2, num_node_p_switch=3, num_gpu_p_node=8, mem_p_node=130), schedule='horus'),
    'horus_early_stop': dict(frame=_zs(lambda: tg.frame_gen(300, 12, 60)), flags=dict(num_switch=3, num_node_p_switch=2, num_gpu_p_node=4), schedule='horus'),
    'horus_gen300': dict(frame=_zs(lambda: tg.frame_gen(300, 11, 150)), flags=dict(num_switch=2, num_node_p_switch=4, num_gpu_p_node=8), schedule='horus', big=True),
    'horus_dense': dict(frame=_zs(lambda: tg.frame_gen(300, 5, 30)), flags=dict(num_switch=2, num_node_p_switch=4, num_gpu_p_node=8), schedule='horus', num_buffer=8, big=True),
    'horus_probe2k': dict(frame=_zs(lambda: tg.frame_gen(2000, 1, 2000)), flags=C4328, schedule='horus', big=True),
    # --schedule gandiva --scheme gandiva (schedule_fifo + horus_placement with gandiva_score + time_slice_check), zero-spread traces
    'gandiva_probe100': dict(frame=_zs(tg.frame_probe100), flags=C148, schedule='gandiva'),
    'gandiva_racks': dict(frame=_zs(tg.frame_probe100), flags=dict(num_switch=2, num_node_p_switch=2, num_gpu_p_node=8), schedule='gandiva'),
    'gandiva_multi_node': dict(frame=_zs(_multi_node), flags=dict(num_switch=2, num_node_p_switch=2, num_gpu_p_node=4), schedule='gandiva'),
    'gandiva_gpu_cap16': dict(frame=_zs(lambda: tg.frame_gen(120, 7, 150)), flags=dict(num_switch=1, num_node_p_switch=8, num_gpu_p_node=8, gpu_memory_capacity=12), schedule='gandiva'),
    'gandiva_ties': dict(frame=_zs(_ties), flags=dict(num_switch=1, num_node_p_switch=2, num_gpu_p_node=8), schedule='gandiva'),
    'gandiva_cluster_spec': dict(frame=_zs(lambda: tg.frame_gen(150, 9, 400)), flags=dict(cluster_spec='@examples/cluster_spec_2x8x4.csv'), schedule='gandiva', big=True),
    'gandiva_gen300': dict(frame=_zs(lambda: tg.frame_gen(300, 11, 150)), flags=dict(num_switch=2, num_node_p_switch=4, num_gpu_p_node=8), schedule='gandiva', big=True),
    'gandiva_probe2k': dict(frame=_zs(lambda: tg.frame_gen(2000, 1, 2000)), flags=C4328, schedule='gandiva', big=True),
    # the same two schedules over --scheme yarn (ms_yarn_placement never reads utilisation: traces keep their spread)
    'horusyarn_probe100': dict(frame=tg.frame_probe100, flags=C148, schedule='horus', scheme='yarn'),
    'horusyarn_big_mem_leak': dict(frame=_big_mem, flags=dict(num_switch=1, num_node_p_switch=3, num_gpu_p_node=4, num_cpu_p_node=64, mem_p_node=256), schedule='horus', scheme='yarn', num_buffer=3),
    'horusyarn_cluster_spec': dict(frame=lambda: tg.frame_gen(150, 9, 400), flags=dict(cluster_spec='@examples/cluster_spec_2x8x4.csv'), schedule='horus', scheme='yarn', big=True),
    'horusyarn_dense': dict(frame=lambda: tg.frame_gen(300, 5, 30), flags=dict(num_switch=2, num_node_p_switch=4, num_gpu_p_node=8), schedule='horus', scheme='yarn', big=True),
    'horusyarn_probe2k': dict(frame=lambda: tg.frame_gen(2000, 1, 2000), flags=C4328, schedule='horus', scheme='yarn', big=True),
    'gandivayarn_probe100': dict(frame=tg.frame_probe100, flags=C148, schedule='gandiva', scheme='yarn'),
    'gandivayarn_multi_node': dict(frame=_multi_node, flags=dict(num_switch=2, num_node_p_switch=2, num_gpu_p_node=4), schedule='gandiva', scheme='yarn'),
    'gandivayarn_cluster_spec': dict(frame=lambda: tg.frame_gen(150, 9, 400), flags=dict(cluster_spec='@examples/cluster_spec_2x8x4.csv'), schedule='gandiva', scheme='yarn', big=True),
    'gandivayarn_dense': dict(frame=lambda: tg.frame_gen(300, 5, 30), flags=dict(num_switch=2, num_node_p_switch=4, num_gpu_p_node=8), schedule='gandiva', scheme='yarn', big=True),
    'gandivayarn_probe2k': dict(frame=lambda: tg.frame_gen(2000, 1, 2000), flags=C4328, schedule='gandiva', scheme='yarn', big=True),
}


def _pack_edges():
    # zero and equal utilisations (CompareAbleByUtilization.__lt__ returns False for a falsy utilisation, base_factory.py:8-12),
    # batches of simultaneous arrivals, a task wider than a node (always leaks, node.py:200-221), memory above the cap margin,
    # used_gpus not divisible by gpu_per_container, long jobs that cross several time slices
    rows = []
    t = 0.0
    for i in range(60):
        g, gpc = [(1, 1), (2, 1), (2, 2), (4, 2), (3, 2), (8, 4), (8, 1), (6, 3), (4, 4), (12, 4)][i % 10]
        ua = [0.0, 37.5, 37.5, 80.0, 12.25, 0.0, 55.0, 37.5, 99.0, 20.0][(i * 7) % 10]
        rows.append(dict(normalized_time=t, minutes=float([3, 40, 7.5, 250, 12, 1, 90, 5, 420, 33][(i * 3) % 10]), used_gpus=float(g), gpu_per_container=gpc,
                         gpu_utilization_avg=ua, gpu_utilization_max=ua, memory_avg=2e9,
                         memory_max=int([3e9, 9e9, 15e9, 33.9e9, 5e9, 20e9, 1e9, 12e9, 7e9, 40e9][(i * 9) % 10])))
        if i % 4 != 3:
            t += [0.0, 12000.0, 30000.0][i % 3]
    rows.append(dict(normalized_time=t + 4e6, minutes=2.0, used_gpus=1.0, gpu_per_container=1, gpu_utilization_avg=5.0, gpu_utilization_max=5.0))
    return tg.frame_rows(rows)


CASES.update({
    'horus_edges': dict(frame=_pack_edges, flags=dict(num_switch=2, num_node_p_switch=2, num_gpu_p_node=4), schedule='horus', num_buffer=4),
    'horus_edges_1node': dict(frame=_pack_edges, flags=dict(num_switch=1, num_node_p_switch=1, num_gpu_p_node=8), schedule='horus', num_buffer=1),
    'gandiva_edges': dict(frame=_pack_edges, flags=dict(num_switch=2, num_node_p_switch=2, num_gpu_p_node=4), schedule='gandiva'),
    'horusyarn_edges': dict(frame=_pack_edges, flags=dict(num_switch=2, num_node_p_switch=2, num_gpu_p_node=4), schedule='horus', scheme='yarn', num_buffer=4),
    'gandivayarn_edges': dict(frame=_pack_edges, flags=dict(num_switch=1, num_node_p_switch=3, num_gpu_p_node=4), schedule='gandiva', scheme='yarn'),
})


# --schedule horus+ (k-means queues): the reference is run with injected k-means draws (oracle/ref_runner.py _INJECT, seed below)
CASES.update({
    'horusplus_probe100_k3': dict(frame=_zs(tg.frame_probe100), flags=C148, schedule='horus+', num_queue=3, inject_seed=1),
    'horusplus_racks_k2': dict(frame=_zs(tg.frame_probe100), flags=dict(num_switch=2, num_node_p_switch=2, num_gpu_p_node=8), schedule='horus+', num_queue=2, inject_seed=5, num_buffer=15),
    'horusplus_ties_k3': dict(frame=_zs(_ties), flags=dict(num_switch=1, num_node_p_switch=2, num_gpu_p_node=8), schedule='horus+', num_queue=3, inject_seed=9),
    'horusplus_edges_k3': dict(frame=_pack_edges, flags=dict(num_switch=2, num_node_p_switch=2, num_gpu_p_node=4), schedule='horus+', num_queue=3, inject_seed=4, num_buffer=4),
    'horusplus_gpu_cap16_k5': dict(frame=_zs(lambda: tg.frame_gen(120, 7, 150)), flags=dict(num_switch=1, num_node_p_switch=8, num_gpu_p_node=8, gpu_memory_capacity=12), schedule='horus+', num_queue=5, inject_seed=7),
    'horusplus_dense_k3': dict(frame=_zs(lambda: tg.frame_gen(300, 5, 30)), flags=dict(num_switch=2, num_node_p_switch=4, num_gpu_p_node=8), schedule='horus+', num_queue=3, inject_seed=1, num_buffer=15, big=True),
    'horusplusyarn_probe100_k3': dict(frame=tg.frame_probe100, flags=C148, schedule='horus+', scheme='yarn', num_queue=3, inject_seed=2),
    'horusplusyarn_dense_k4': dict(frame=lambda: tg.frame_gen(300, 5, 30), flags=dict(num_switch=2, num_node_p_switch=4, num_gpu_p_node=8), schedule='horus+', scheme='yarn', num_queue=4, inject_seed=3, big=True),
})
CASES['horusplus_probe2k_k3'] = dict(frame=_zs(lambda: tg.frame_gen(2000, 1, 2000)), flags=C4328, schedule='horus+', num_queue=3, inject_seed=1, num_buffer=15, big=True)
CASES['horus_probe10k'] = dict(frame=_zs(lambda: tg.frame_gen(10000, 2, 10000)), flags=C4328, schedule='horus', big=True, huge=True)   # 72 min of reference time
CASES['gandiva_probe10k'] = dict(frame=_zs(lambda: tg.frame_gen(10000, 2, 10000)), flags=C4328, schedule='gandiva', big=True, huge=True)
CASES['horusyarn_probe10k'] = dict(frame=lambda: tg.frame_gen(10000, 2, 10000), flags=C4328, schedule='horus', scheme='yarn', big=True, huge=True)
CASES['gandivayarn_probe10k'] = dict(frame=lambda: tg.frame_gen(10000, 2, 10000), flags=C4328, schedule='gandiva', scheme='yarn', big=True, huge=True)
CASES['horusplus_probe10k_k3'] = dict(frame=_zs(lambda: tg.frame_gen(10000, 2, 10000)), flags=C4328, schedule='horus+', num_queue=3, inject_seed=1, num_buffer=15, big=True, huge=True)


# ---- legacy event loops (dead code in the reference, executed unmodified by oracle/ref_legacy_runner.py under shim globals):
# sjf / shortest / shortest-gpu over the live yarn fit, dlas-gpu / dlas with count-based admission.  `queue_limit` in GPU-ticks / ticks.
LEGACY = ('sjf', 'shortest', 'shortest-gpu', 'dlas-gpu', 'dlas')
_S248 = dict(num_switch=2, num_node_p_switch=4, num_gpu_p_node=8)
_S164 = dict(num_switch=1, num_node_p_switch=6, num_gpu_p_node=4)
CASES.update({
    'sjf_dense': dict(frame=lambda: tg.frame_gen(300, 5, 30), flags=_S248, schedule='sjf'),
    'sjf_dense2': dict(frame=lambda: tg.frame_gen(500, 6, 60), flags=_S164, schedule='sjf', big=True),
    'sjf_ties': dict(frame=_ties, flags=dict(num_switch=1, num_node_p_switch=2, num_gpu_p_node=8), schedule='sjf'),
    'sjf_multi_node': dict(frame=_multi_node, flags=dict(num_switch=2, num_node_p_switch=2, num_gpu_p_node=4), schedule='sjf'),
    'sjf_big_mem_leak': dict(frame=_big_mem, flags=dict(num_switch=1, num_node_p_switch=3, num_gpu_p_node=4, num_cpu_p_node=64, mem_p_node=256), schedule='sjf'),
    'sjf_kat6': dict(frame=_kat6, flags=dict(num_switch=1, num_node_p_switch=1, num_gpu_p_node=8), schedule='sjf'),
    'sjf_probe2k': dict(frame=lambda: tg.frame_gen(2000, 1, 2000), flags=C4328, schedule='sjf', big=True),
    'sjf_loaded3k': dict(frame=lambda: tg.frame_gen(3000, 4, 500), flags=C4328, schedule='sjf', big=True, huge=True),
    'sjf_probe10k': dict(frame=lambda: tg.frame_gen(10000, 2, 10000), flags=C4328, schedule='sjf', big=True, huge=True),   # BASELINE config C2
    'shortest_dense': dict(frame=lambda: tg.frame_gen(300, 5, 30), flags=_S248, schedule='shortest', big=True),
    'shortest_light': dict(frame=lambda: tg.frame_gen(400, 8, 400), flags=_S248, schedule='shortest', big=True),
    'shortest_multi_node': dict(frame=_multi_node, flags=dict(num_switch=2, num_node_p_switch=2, num_gpu_p_node=4), schedule='shortest'),
    'shortestgpu_dense2': dict(frame=lambda: tg.frame_gen(500, 6, 60), flags=_S164, schedule='shortest-gpu', big=True),
    'shortestgpu_ties': dict(frame=_ties, flags=dict(num_switch=1, num_node_p_switch=2, num_gpu_p_node=8), schedule='shortest-gpu'),
    'dlasgpu_dense': dict(frame=lambda: tg.frame_gen(300, 5, 30), flags=_S248, schedule='dlas-gpu', queue_limit=(30, 60, 150), big=True),
    'dlasgpu_dense2_q2': dict(frame=lambda: tg.frame_gen(500, 6, 60), flags=_S164, schedule='dlas-gpu', queue_limit=(8,), big=True),
    'dlasgpu_light_q6': dict(frame=lambda: tg.frame_gen(400, 8, 400), flags=_S248, schedule='dlas-gpu', queue_limit=(5, 9, 14, 20, 33), big=True),
    'dlasgpu_ties': dict(frame=_ties, flags=dict(num_switch=1, num_node_p_switch=2, num_gpu_p_node=8), schedule='dlas-gpu', queue_limit=(30, 60, 150)),
    'dlasgpu_multi_node': dict(frame=_multi_node, flags=dict(num_switch=2, num_node_p_switch=2, num_gpu_p_node=4), schedule='dlas-gpu', queue_limit=(30, 60, 150)),   # stale end_jobs on a start event (run_sim.py:706-717)
    'dlasgpu_kat6': dict(frame=_kat6, flags=dict(num_switch=1, num_node_p_switch=1, num_gpu_p_node=8), schedule='dlas-gpu', queue_limit=(30, 60, 150)),
    'dlasgpu_probe2k': dict(frame=lambda: tg.frame_gen(2000, 1, 2000), flags=C4328, schedule='dlas-gpu', queue_limit=(30, 60, 150), big=True),
    'dlasgpu_loaded3k': dict(frame=lambda: tg.frame_gen(3000, 4, 500), flags=C4328, schedule='dlas-gpu', queue_limit=(30, 60, 150), big=True, huge=True),
    'dlasgpu_probe60k': dict(frame=lambda: tg.frame_gen(60000, 3, 60000), flags=C4328, schedule='dlas-gpu', queue_limit=(30, 60, 150), big=True, huge=True),   # BASELINE config C3
    'dlas_dense': dict(frame=lambda: tg.frame_gen(300, 5, 30), flags=_S248, schedule='dlas', queue_limit=(30, 60, 150), big=True),
    'dlas_multi_node': dict(frame=_multi_node, flags=dict(num_switch=2, num_node_p_switch=2, num_gpu_p_node=4), schedule='dlas', queue_limit=(8, 12)),
    'dlas_probe2k': dict(frame=lambda: tg.frame_gen(2000, 1, 2000), flags=C4328, schedule='dlas', queue_limit=(30, 60, 150), big=True),
})


# ---- random traces and cluster shapes, recorded from the reference by `python oracle/make_golden.py --random` into
# tests/golden/random_cases.json.gz (tests/test_oracle_vs_live_reference.py; tests/test_gpu_random.py draws from the same generator)
RANDOM_GOLD = 'random_cases.json.gz'
RANDOM_PACK_COMBOS = [('horus', 'horus'), ('gandiva', 'gandiva'), ('horus+', 'horus+'), ('horus', 'yarn'), ('gandiva', 'yarn'), ('horus+', 'yarn')]
RANDOM_FIFO = list(range(100, 112))
RANDOM_PACK = [(200 + 3 * i + j, combo) for i, combo in enumerate(RANDOM_PACK_COMBOS) for j in range(2)]
RANDOM_LEGACY = [(300 + 5 * i + j, sched) for i, sched in enumerate(LEGACY) for j in range(2)]


def random_case(seed):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(20, 90))
    flags = dict(num_switch=int(rng.integers(1, 3)), num_node_p_switch=int(rng.integers(1, 5)),
                 num_gpu_p_node=int(rng.choice([2, 4, 8])), num_cpu_p_node=int(rng.choice([24, 48, 128])),
                 mem_p_node=int(rng.choice([120, 256, 512])), gpu_memory_capacity=int(rng.choice([8, 16, 32])))
    g = rng.choice([1, 2, 3, 4, 6, 8, 16], n)
    gpc = np.array([int(rng.choice([c for c in (1, 2, 3, 4, 8) if c <= x])) for x in g])
    rows = [dict(normalized_time=float(t), minutes=float(m), used_gpus=float(a), gpu_per_container=int(b),
                 memory_max=int(mm), gpu_utilization_avg=float(u), gpu_utilization_max=float(min(100, u + 10)))
            for t, m, a, b, mm, u in zip(np.sort(rng.uniform(0, 6e5, n)).round(-3 if seed % 2 else 0), rng.uniform(0.5, 60, n), g, gpc,
                                         rng.uniform(5e8, 1.9e10, n), rng.uniform(1, 90, n))]
    return tg.frame_rows(rows), flags


def random_pack_case(seed, sched, scheme):
    """Trace, flags and (look-ahead, queue count, k-means injection seed) of a random pack-family case; over the pack placement
    the trace has zero utilisation spread (the reference's draws return their mean)."""
    df, flags = random_case(seed)
    if scheme != 'yarn':
        df = df.copy(); df['gpu_utilization_max'] = df['gpu_utilization_avg']
    rng = np.random.default_rng(seed + 7)
    k = int(rng.integers(1, 8)); kq = int(rng.integers(1, 5)); inj = int(rng.integers(1, 1000))
    return df, flags, k, kq, inj


def random_legacy_queue_limit(seed):
    rng = np.random.default_rng(seed + 11)
    return tuple(int(x) for x in np.cumsum(rng.integers(5, 60, int(rng.integers(1, 4)))))   # 2 .. 4 queues


def random_key(family, seed, *rest):
    return '/'.join((family, str(seed)) + rest)
