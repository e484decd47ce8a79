"""Pin the CPU oracle (oracle/metis_oracle.py) to outputs of the unmodified reference.

The golden files were produced by tests/golden/make_golden.py, which imports
/root/reference in the build container.  Everything here is exact: candidate
order, partitions, strategies and the bits of every fp64 cost.
"""
import os
import random

import pytest

from conftest import C1_DIR, golden_rows, load_golden
from golden_units import load_units
from oracle import metis_oracle as orc


def _oracle_inputs(root, profile_sub, file_order, num_layers, hidden, seq, vocab):
    cluster = orc.OracleCluster(os.path.join(root, 'hostfile'), os.path.join(root, 'clusterfile.json'))
    profile, types = orc.load_profile_dir(os.path.join(root, profile_sub), file_order)
    model = orc.OracleModel(num_layers, hidden, seq, vocab, profile['model']['parameters'])
    return cluster, profile, types, model


def _run_het(meta, root, profile_sub, w):
    cluster, profile, _, model = _oracle_inputs(root, profile_sub, meta['file_order'], w['L'], w['hidden'],
                                                w['seq'], w['vocab'])
    seqs = [tuple(s) for s in meta['node_sequences']]
    return orc.het_search(profile, cluster, model, seqs, w['gbs'], w['L'], w['variance'], w['mpl'],
                          w['max_tp'], w['max_bs'])


def _same(cands, gold):
    assert len(cands) == len(gold)
    for c, g in zip(cands, gold):
        ordinal, step, _ns, groups, strategies, batches, part, nrep, cost = c
        assert (ordinal, step, groups, strategies, batches, part, nrep) == (g[0], g[1], g[3], g[4], g[5], g[6], g[7])
        assert cost == g[8], (ordinal, step, cost.hex(), g[8].hex())


def test_fsum_is_builtin_sum():
    rng = random.Random(3)
    for _ in range(3000):
        xs = [rng.uniform(-1, 1) * 10 ** rng.randint(-8, 8) for _ in range(rng.randint(0, 40))]
        if rng.random() < 0.3:
            xs = [rng.randint(0, 5) for _ in range(rng.randint(0, 3))] + xs
        if rng.random() < 0.2 and xs:
            xs[rng.randrange(len(xs))] = 0
        assert orc.fsum(xs) == sum(xs)


def test_c1_het_kat1():
    meta, arr = load_golden('c1_het')
    w = dict(L=10, hidden=4096, seq=1024, vocab=51200, gbs=128, variance=1, mpl=4, max_tp=4, max_bs=4)
    cands, counters = _run_het(meta, C1_DIR, 'profile_data_samples', w)
    assert counters['A'] == meta['counters']['A'] == 32
    assert counters['C'] == 19
    _same(cands, golden_rows(arr))
    best = min(cands, key=lambda c: c[8])
    assert best[8] == 621.8881853975784 and best[3] == [64] and best[4] == [(64, 1)] and best[6] == [0, 10]


def test_c1_homo_kat2():
    meta, arr = load_golden('c1_homo')
    cluster, profile, types, model = _oracle_inputs(C1_DIR, 'profile_data_samples', meta['file_order'],
                                                    10, 4096, 1024, 51200)
    out, counters = orc.homo_search(profile, cluster, model, types[0], 128, 4)
    assert counters['yielded'] == meta['yielded'] == 345
    assert counters['matched'] == 98 and counters['costed'] == meta['costed'] == 53
    assert [list(p) for p, _ in out] == arr['plan'].tolist()
    assert [c for _, c in out] == arr['cost'].tolist()


@pytest.mark.parametrize('name', ['c2_het16', 'c2_v100', 'mix32', 'het32_tight', 'sweep_n8_t1', 'sweep_n16_t2_v0',
                                  'long_profile', 'q10_big_first'])
def test_synthetic_het(name, workload_dir):
    meta, arr = load_golden(name)
    w, root, digest = workload_dir(name)
    assert digest == meta['inputs_sha256'], 'synthetic generator drifted from the golden inputs'
    cfg = dict(L=w.num_layers, hidden=w.hidden_size, seq=w.sequence_length, vocab=w.vocab_size, gbs=w.gbs,
               variance=w.variance, mpl=w.max_permute_len, max_tp=w.max_tp, max_bs=w.max_bs)
    cands, counters = _run_het(meta, root, 'profile', cfg)
    for k in ('A', 'B', 'runs', 'C'):
        assert counters[k] == meta['counters'][k], k
    _same(cands, golden_rows(arr))


def test_fatal_keyerror(workload_dir):
    meta, arr = load_golden('fatal_gbs96')
    w, root, _ = workload_dir('fatal_gbs96')
    cluster, profile, _, model = _oracle_inputs(root, 'profile', meta['file_order'], w.num_layers,
                                                w.hidden_size, w.sequence_length, w.vocab_size)
    with pytest.raises(KeyError) as err:
        orc.het_search(profile, cluster, model, [tuple(s) for s in meta['node_sequences']], w.gbs,
                       w.num_layers, w.variance, w.max_permute_len, w.max_tp, w.max_bs)
    assert meta['fatal'][1] == 'KeyError' and str(err.value) == meta['fatal'][2]


@pytest.mark.parametrize('name', ['q10_small_first', 'q10_small_first_t1'])
def test_fatal_indexerror_unequal_nodes(name, workload_dir):
    """Quirk Q10 with node 0 SMALLER than the others: the rank list of the memory model is too short and the
    reference dies with IndexError at the first stage that reaches past it (load_balancer.py:36)."""
    meta, arr = load_golden(name)
    w, root, _ = workload_dir(name)
    cluster, profile, _, model = _oracle_inputs(root, 'profile', meta['file_order'], w.num_layers,
                                                w.hidden_size, w.sequence_length, w.vocab_size)
    with pytest.raises(IndexError) as err:
        orc.het_search(profile, cluster, model, [tuple(s) for s in meta['node_sequences']], w.gbs,
                       w.num_layers, w.variance, w.max_permute_len, w.max_tp, w.max_bs)
    assert meta['fatal'][1] == 'IndexError' and str(err.value) == meta['fatal'][2]


@pytest.fixture(scope='module')
def units():
    return load_units()


def test_units_device_groups(units):
    for case in units['device_groups']:
        rows = orc.device_group_rows(case['stages'], case['ndev'], case['variance'], case['mpl'])
        assert rows == case['rows'], case


def test_units_balancer(units):
    for case in units['balancer']:
        lc = [float.fromhex(x) for x in case['lc']]
        capa = [float.fromhex(x) for x in case['capa']]
        assert orc.layer_compute_balance(case['S'], case['L'], capa, lc) == case['part']


def test_units_adjust(units):
    for case in units['adjust']:
        out = orc.adjust_compute_performance([float.fromhex(x) for x in case['c']], case['mc'],
                                             [float.fromhex(x) for x in case['md']])
        want = None if case['out'] is None else [float.fromhex(x) for x in case['out']]
        assert out == want


@pytest.mark.parametrize('name', ['c3_homo64_mpl4', 'sweep_n8_t1'])
def test_synthetic_homo(name, workload_dir):
    meta, arr = load_golden(name + '_homo')
    w, root, digest = workload_dir(name)
    assert digest == meta['inputs_sha256']
    cluster, profile, types, model = _oracle_inputs(root, 'profile', meta['file_order'], w.num_layers,
                                                    w.hidden_size, w.sequence_length, w.vocab_size)
    out, counters = orc.homo_search(profile, cluster, model, types[0], w.gbs, w.max_tp)
    assert counters['yielded'] == meta['yielded'] and counters['costed'] == meta['costed']
    assert [list(p) for p, _ in out] == arr['plan'].tolist()
    assert [c for _, c in out] == arr['cost'].tolist()
