"""Randomised differential test: oracle/cpu_sim.c vs the UNMODIFIED reference on random traces / cluster shapes.
The reference's files for every seed listed in oracle/golden_cases.py (RANDOM_*) were recorded from live runs by
`python oracle/make_golden.py --random` into tests/golden/random_cases.json.gz; the oracle is run here and compared with
them byte for byte.  Complements the fixed golden cases."""
import gzip
import io
import json
import os

import pandas as pd
import pytest

import cpu_sim
import golden_cases
import goldutil


@pytest.fixture(scope='module')
def recorded():
    with gzip.open(os.path.join(goldutil.GOLD, golden_cases.RANDOM_GOLD), 'rt') as f:
        return json.load(f)


def _trace(df, rec):
    """The trace as the reference read it: the CSV text, checked against the sha256 recorded with the reference's files."""
    txt = df.to_csv(index=False)
    assert goldutil.sha(txt) == rec['trace_sha256'], 'the random case generator drifted from the recording'
    return cpu_sim.prepare_trace(pd.read_csv(io.StringIO(txt)))


def test_oracle_equals_live_reference_on_random_cases(recorded):
    for seed in golden_cases.RANDOM_FIFO:
        ref = recorded[golden_cases.random_key('fifo', seed)]
        df, flags = golden_cases.random_case(seed)
        tr = _trace(df, ref)
        res = cpu_sim.run_fifo_yarn(cpu_sim.make_cluster(**flags), tr)
        assert ref['job_csv'] is not None, seed
        assert cpu_sim.format_job_csv(tr, res) == ref['job_csv'], seed
        assert cpu_sim.format_cluster_csv(res) == ref['cluster_csv'], seed


# ---- the pack family: horus / horus+ / gandiva over the pack placement (zero utilisation spread: the reference's draws return
# their mean) and over yarn (real spread); horus+ with its k-means draws injected (ref_runner._INJECT)
def test_pack_oracle_equals_live_reference_on_random_cases(recorded):
    for seed, (sched, scheme) in golden_cases.RANDOM_PACK:
        ref = recorded[golden_cases.random_key('pack', seed, sched, scheme)]
        df, flags, k, kq, inj = golden_cases.random_pack_case(seed, sched, scheme)
        tr = _trace(df, ref)
        try:
            res = cpu_sim.run_pack(cpu_sim.make_cluster(**flags), tr, sched, k, scheme=('yarn' if scheme == 'yarn' else None),
                                   num_queue=kq, inject_seed=inj)
        except RuntimeError:   # the oracle says the reference raises on this input
            assert ref['returncode'] != 0 or ref['job_csv'] is None or ref['stderr_has_error'], (seed, sched, scheme)
            continue
        assert ref['job_csv'] is not None, (seed, sched, scheme)
        assert cpu_sim.format_job_csv(tr, res) == ref['job_csv'], (seed, sched, scheme)
        assert cpu_sim.format_cluster_csv(res) == ref['cluster_csv'], (seed, sched, scheme)


# ---- the legacy event loops: the reference's dead code run unmodified under the shim globals (oracle/ref_legacy_runner.py)
def test_legacy_oracle_equals_live_reference_on_random_cases(recorded):
    for seed, sched in golden_cases.RANDOM_LEGACY:
        ref = recorded[golden_cases.random_key('legacy', seed, sched)]
        df, flags = golden_cases.random_case(seed)
        tr = _trace(df, ref)
        ql = golden_cases.random_legacy_queue_limit(seed)
        cluster = cpu_sim.make_cluster(**flags)
        res, count = cpu_sim.run_legacy(cluster, tr, sched, ql)
        assert ref['job_csv'] is not None and ref['cluster_csv'] is not None, (seed, sched)
        assert cpu_sim.format_legacy_job_csv(tr, res, count) == ref['job_csv'], (seed, sched)
        assert cpu_sim.format_legacy_cluster_csv(res, cluster, count) == ref['cluster_csv'], (seed, sched)
