"""CPU checks of the device evaluator's *logic* (tests/hostsim = g++ build of
metis_b200/csrc/metis_eval.cuh) plus the host flattening / C++ enumerator, against the golden
files produced by the unmodified reference.  The GPU parity tests proper are in
test_gpu_parity.py (-m gpu); this file exists because the build container has no GPU.
"""
import gzip
import json
import os

import numpy as np
import pytest

import hostsim_util as hs
from conftest import C1_DIR, GOLDEN, assert_candidates_equal, device_columns, golden_rows, load_golden
from golden_units import load_units
from metis_b200 import flatten, native


def _lib_or_skip():
    try:
        return native.load_library()
    except native.MetisNativeError as e:
        pytest.skip(str(e))


def _search(meta, root, profile_sub, num_layers, hidden, seq, vocab, gbs, variance, mpl, max_tp, max_bs,
            **kw):
    lib = _lib_or_skip()
    cluster, profile, _types, cfg = hs.load_inputs(root, profile_sub, meta['file_order'], num_layers, hidden, seq, vocab)
    seqs = [tuple(s) for s in meta['node_sequences']]
    problem = flatten.build_problem(profile, cluster, cfg, gbs, max_tp, max_bs, seqs)
    space = flatten.build_plan_space(len(seqs), cluster.get_total_num_devices(), gbs, num_layers, variance, mpl, lib)
    return problem, space, hs.host_het_search(problem, space, **kw)


def _compare(cands, gold):
    assert len(cands) == len(gold)
    for c, g in zip(cands, gold):
        assert c[:8] == g[:8], (c, g)
        assert c[8] == g[8], (c[0], c[1], c[8].hex(), g[8].hex())


def test_c1_het():
    meta, arr = load_golden('c1_het')
    problem, space, (rec, det, summary) = _search(meta, C1_DIR, 'profile_data_samples', 10, 4096, 1024, 51200,
                                                  128, 1, 4, 4, 4)
    assert space.num_plans == meta['counters']['A'] == 32
    assert summary.num_records == 19 and summary.num_partition_calls == meta['counters']['B']
    _compare(hs.unpack_candidates(rec, det, space), golden_rows(arr))
    assert summary.best.cost == 621.8881853975784 and summary.best.ordinal == 7


@pytest.mark.parametrize('mode', [0, 1, 2, 3, 4], ids=['sequential_run', 'first_task_then_chain', 'chain_only',
                                                   'chain_only_reversed_par_sections', 'first_task_then_replay'])
@pytest.mark.parametrize('name', ['c2_het16', 'c2_v100', 'mix32', 'het32_tight', 'sweep_n8_t1', 'sweep_n16_t2_v0',
                                  'long_profile', 'q10_big_first'])
def test_synthetic(name, mode, workload_dir):
    meta, arr = load_golden(name)
    w, root, _ = workload_dir(name)
    problem, space, (rec, det, summary) = _search(meta, root, 'profile', w.num_layers, w.hidden_size,
                                                  w.sequence_length, w.vocab_size, w.gbs, w.variance,
                                                  w.max_permute_len, w.max_tp, w.max_bs, mode=mode)
    c = meta['counters']
    assert space.num_plans == c['A']
    assert (summary.num_partition_calls, summary.num_balancer_runs, summary.num_records) == (c['B'], c['runs'], c['C'])
    assert summary.fatal_ordinal == 2 ** 64 - 1
    gold = golden_rows(arr)
    _compare(hs.unpack_candidates(rec, det, space), gold)
    best = min(gold, key=lambda g: (g[8], g[0], g[1]))
    assert (summary.best.cost, summary.best.ordinal, summary.best.step) == (best[8], best[0], best[1])


def test_sharded_union_equals_whole(workload_dir):
    meta, arr = load_golden('c2_v100')
    w, root, _ = workload_dir('c2_v100')
    got = []
    for rank in range(3):
        problem, space, (rec, det, _s) = _search(meta, root, 'profile', w.num_layers, w.hidden_size,
                                                 w.sequence_length, w.vocab_size, w.gbs, w.variance,
                                                 w.max_permute_len, w.max_tp, w.max_bs, rank=rank, world=3, tile=64)
        got += hs.unpack_candidates(rec, det, space)
    got.sort(key=lambda c: (c[0], c[1]))
    _compare(got, golden_rows(arr))


def test_fatal_keyerror(workload_dir):
    meta, _ = load_golden('fatal_gbs96')
    w, root, _ = workload_dir('fatal_gbs96')
    _, _, (_rec, _det, summary) = _search(meta, root, 'profile', w.num_layers, w.hidden_size, w.sequence_length,
                                          w.vocab_size, w.gbs, w.variance, w.max_permute_len, w.max_tp, w.max_bs)
    assert summary.fatal_ordinal == meta['fatal'][0]
    assert summary.fatal_code == 1 and summary.fatal_aux == (0 << 16 | 3)     # 'tp1_bs3'


@pytest.mark.parametrize('mode', [0, 1, 2])
@pytest.mark.parametrize('name', ['q10_small_first', 'q10_small_first_t1'])
def test_fatal_indexerror_unequal_nodes(name, mode, workload_dir):
    """Node 0 smaller than the others (quirk Q10): the reference aborts with IndexError at the first plan whose stage
    reaches past the too-short rank list; the device reports that plan and the INDEX code."""
    meta, _ = load_golden(name)
    w, root, _ = workload_dir(name)
    _, _, (_rec, _det, summary) = _search(meta, root, 'profile', w.num_layers, w.hidden_size, w.sequence_length,
                                          w.vocab_size, w.gbs, w.variance, w.max_permute_len, w.max_tp, w.max_bs, mode=mode)
    assert summary.fatal_ordinal == meta['fatal'][0] and summary.fatal_code == 3


@pytest.fixture(scope='module')
def units():
    return load_units()


def test_units_enumerator(units):
    lib = _lib_or_skip()
    for case in units['device_groups']:
        rows = flatten.enumerate_device_groups(case['stages'], case['ndev'], case['variance'], case['mpl'], lib)
        want = np.array(case['rows'], dtype=np.int64).reshape(-1, case['stages'])
        assert rows.shape == want.shape, case
        assert ((1 << rows.astype(np.int64)) == want).all(), case


def test_enumerator_vs_oracle_grid():
    """The C++ enumerator (count-vector search with exact feasibility, slice-based merging) against the
    oracle's restatement of gen_dgroups_for_stages_with_variance over a grid of cluster sizes, stage counts,
    variances and max_permute_len - including spaces the unit fixtures do not hold (256 devices, variance 0 / 0.5)."""
    from oracle import metis_oracle as orc
    lib = _lib_or_skip()
    checked = rows_total = 0
    for ndev in (4, 8, 16, 32, 64, 128, 256):
        for stages in sorted({1, 2, 3, 5, 7, 8, 12, 16, 24, 31, 32, 48, 64, 100, 128, ndev - 1, ndev, ndev + 1}):
            for variance in (0, 0.5, 1):
                for mpl in (1, 2, 4, 6):
                    if stages < 1 or (variance != 1 and (stages > 24 or ndev > 64)) or (mpl == 6 and ndev > 64 and stages > 40):
                        continue                      # keep the Python side to seconds
                    rows = flatten.enumerate_device_groups(stages, ndev, variance, mpl, lib)
                    want = orc.device_group_rows(stages, ndev, variance, mpl)
                    assert rows.shape[0] == len(want), (ndev, stages, variance, mpl)
                    if want:
                        assert ((1 << rows.astype(np.int64)) == np.array(want, dtype=np.int64)).all(), (ndev, stages, variance, mpl)
                    checked += 1
                    rows_total += len(want)
    assert checked > 400 and rows_total > 50000


def test_units_balancer(units):
    by_l = {}
    for case in units['balancer']:
        by_l.setdefault((case['L'], tuple(case['lc'])), []).append(case)
    for (L, lc_hex), cases in by_l.items():
        lc = [float.fromhex(x) for x in lc_hex]
        got = hs.host_layer_balance([[float.fromhex(x) for x in c['capa']] for c in cases], lc, L)
        for g, c in zip(got, cases):
            assert g == c['part'], c


@pytest.mark.parametrize('name', ['c3_homo64_mpl4', 'c4_het128', 'sweep_n32_t4'])
def test_full_size_spaces_on_host(name, workload_dir):
    """8.3e4-plan C3 space (all candidates) and the 4.5e6-plan C4 space (reference-sampled ordinals)."""
    meta, arr = load_golden(name)
    w, root, digest = workload_dir(name)
    assert digest == meta['inputs_sha256']
    problem, space, (rec, det, summary) = _search(meta, root, 'profile', w.num_layers, w.hidden_size,
                                                  w.sequence_length, w.vocab_size, w.gbs, w.variance,
                                                  w.max_permute_len, w.max_tp, w.max_bs)
    assert space.num_plans == meta['counters']['A']
    assert summary.fatal_ordinal == 2 ** 64 - 1
    order = np.lexsort((rec['step'], rec['ordinal']))
    rec, det = rec[order], det[order]
    if 'sample' in arr:
        keep = np.isin(rec['ordinal'].astype(np.int64), arr['sample'])
        rec, det = rec[keep], det[keep]
    else:
        c = meta['counters']
        assert (summary.num_partition_calls, summary.num_balancer_runs, summary.num_records) == (c['B'], c['runs'], c['C'])
    assert_candidates_equal(device_columns(rec, det, arr['dp'].shape[1]), meta, arr)


@pytest.mark.parametrize('name,root_kind', [('c1', 'c1'), ('c3_homo64_mpl4', 'syn'), ('sweep_n8_t1', 'syn')])
def test_homo_cost_on_host(name, root_kind, workload_dir):
    """HomoCostEstimator.get_cost (device code, host build) against the reference's costs."""
    from metis_b200 import api
    from metis_b200.arguments import parse_args
    if root_kind == 'c1':
        meta, arr = load_golden('c1_homo')
        root, sub, L, hid, seq, voc, gbs, max_tp = C1_DIR, 'profile_data_samples', 10, 4096, 1024, 51200, 128, 4
    else:
        meta, arr = load_golden(name + '_homo')
        w, root, _ = workload_dir(name)
        sub, L, hid, seq, voc, gbs, max_tp = 'profile', w.num_layers, w.hidden_size, w.sequence_length, w.vocab_size, w.gbs, w.max_tp
    cluster, profile, types, cfg = hs.load_inputs(root, sub, meta['file_order'], L, hid, seq, voc)
    plans = np.array([[p.dp, p.pp, p.tp, p.mbs, p.gbs] for p in api.UniformPlanGenerator(cluster.get_total_num_devices(), max_tp, gbs)
                      if p.gbs == gbs], dtype=np.int32)
    problem = flatten.build_problem(profile, cluster, cfg, gbs, int(plans[:, 2].max()), int(plans[:, 3].max()),
                                    [tuple(dict.fromkeys(t.name for t in cluster.get_device_types()))])
    cost, status = hs.host_homo_cost(problem, problem.type_names.index(types[0]), plans)
    keep = status != 1
    assert plans[keep].tolist() == arr['plan'].tolist()
    assert cost[keep].tolist() == arr['cost'].tolist()


def _random_workload(rng, idx):
    from metis_b200.workloads import Workload
    types = rng.sample(['A100', 'H100', 'B200', 'V100'], rng.choice([1, 1, 2, 2, 3]))
    per = rng.choice([2, 4, 8])
    nnodes = rng.choice([1, 2, 2, 3, 4]) if per < 8 else rng.choice([1, 2, 3])
    nnodes = max(nnodes, len(types))
    nodes = [(types[(i * len(types)) // nnodes], per) for i in range(nnodes)]      # runs of equal types, like a hostfile
    layers = rng.randint(6, 28)
    memory = {t: rng.choice([6, 10, 16, 24, 40, 80]) for t in types}               # small memories force re-partitioning
    bw = {t: rng.choice([5312500000.0, 2.5e9, 9.0e10]) for t in types}
    return Workload(f'fuzz{idx}', nodes, layers, rng.choice([8, 12, 16, 24, 32, 48, 64]),
                    rng.choice([1024, 4096, 8192]), rng.choice([512, 2048]), rng.choice([30522, 51200]),
                    variance=rng.choice([0, 0.5, 1, 1]), max_permute_len=rng.choice([2, 3, 4, 6]),
                    max_tp=rng.choice([1, 2, 4]), max_bs=rng.choice([1, 2, 4]), bss=(1, 2, 4, 8, 16), seed=idx,
                    memory_gb=memory, intra_bw=bw)


def test_random_small_clusters_vs_oracle(tmp_path):
    """Seeded fuzz: 160 random small clusters (1-3 device types, 2-32 GPUs, odd layer counts and batch sizes, tight
    memories, variance 0 / 0.5 / 1) searched by the device code (host build, all four scheduling modes in turn) and
    by the oracle; every candidate, counter and fp64 cost bit must agree, and a search the oracle aborts with a
    KeyError must report the same plan."""
    import itertools
    import random
    from oracle import metis_oracle as orc
    from metis_b200.workloads import materialize, profile_file_order
    rng = random.Random(20260921)
    done = fatal = candidates = 0
    idx = 0
    while done < 160 and idx < 1600:
        idx += 1
        w = _random_workload(rng, idx)
        root = str(tmp_path / w.name)
        materialize(w, root)
        order = profile_file_order(w)
        cluster, profile, _types, cfg = hs.load_inputs(root, 'profile', order, w.num_layers, w.hidden_size,
                                                       w.sequence_length, w.vocab_size)
        seqs = list(itertools.permutations(w.device_types()))
        ndev = cluster.get_total_num_devices()
        try:
            space = flatten.build_plan_space(len(seqs), ndev, w.gbs, w.num_layers, w.variance, w.max_permute_len)
        except IndexError:
            continue                                   # no stage-1 rows: the reference raises before searching
        if not 1 <= space.num_plans <= 6000:
            continue
        problem = flatten.build_problem(profile, cluster, cfg, w.gbs, w.max_tp, w.max_bs, seqs)
        rec, det, summary = hs.host_het_search(problem, space, mode=done % 4)
        ocl = orc.OracleCluster(os.path.join(root, 'hostfile'), os.path.join(root, 'clusterfile.json'))
        oprof, _ = orc.load_profile_dir(os.path.join(root, 'profile'), order)
        omodel = orc.OracleModel(w.num_layers, w.hidden_size, w.sequence_length, w.vocab_size, oprof['model']['parameters'])
        try:
            want, counters = orc.het_search(oprof, ocl, omodel, seqs, w.gbs, w.num_layers, w.variance,
                                            w.max_permute_len, w.max_tp, w.max_bs)
        except KeyError:
            assert summary.fatal_ordinal != 2 ** 64 - 1 and summary.fatal_code in (1, 2), w
            fatal += 1
            done += 1
            continue
        assert summary.fatal_ordinal == 2 ** 64 - 1, w
        assert (space.num_plans, summary.num_partition_calls, summary.num_balancer_runs, summary.num_records) == \
            (counters['A'], counters['B'], counters['runs'], counters['C']), w
        got = hs.unpack_candidates(rec, det, space)
        assert len(got) == len(want), w
        for g, x in zip(got, want):
            assert (g[0], g[1], g[3], g[4], g[5], g[6], g[7]) == (x[0], x[1], x[3], x[4], x[5], x[6], x[7]), (w, g, x)
            assert g[8] == x[8], (w, g[0], g[1], g[8].hex(), x[8].hex())
        candidates += len(want)
        done += 1
    assert done == 160 and candidates > 2000 and 0 < fatal < 40, (done, fatal, candidates)


@pytest.mark.parametrize('name', ['c2_het16', 'mix32'])
def test_opt_in_corrected_mode(name, workload_dir):
    """SURVEY.md 8(f)-4: with corrected=('Q1', 'Q2') the host drops the mislabelled one-stage blocks and fills the
    between-node bandwidth from the clusterfile's inter_bandwidth; the device code is unchanged.  The result equals
    the oracle run with the same corrections, differs from the strict search, and the strict default still equals
    the golden (other tests)."""
    import itertools
    from oracle import metis_oracle as orc
    meta, arr = load_golden(name)
    w, root, _ = workload_dir(name)
    cluster, profile, _types, cfg = hs.load_inputs(root, 'profile', meta['file_order'], w.num_layers, w.hidden_size,
                                                   w.sequence_length, w.vocab_size)
    seqs = [tuple(s) for s in meta['node_sequences']]
    fix = ('Q1', 'Q2')
    problem = flatten.build_problem(profile, cluster, cfg, w.gbs, w.max_tp, w.max_bs, seqs, corrected=fix)
    space = flatten.build_plan_space(len(seqs), cluster.get_total_num_devices(), w.gbs, w.num_layers, w.variance,
                                     w.max_permute_len, corrected=fix)
    strict = flatten.build_plan_space(len(seqs), cluster.get_total_num_devices(), w.gbs, w.num_layers, w.variance,
                                      w.max_permute_len)
    mislabelled = [b for b in strict.blocks if int(b['label_stage']) != int(b['num_stage'])]
    assert len(seqs) > 1 and len(mislabelled) == len(seqs) - 1            # quirk Q1 in the strict space ...
    assert all(int(b['label_stage']) == int(b['num_stage']) for b in space.blocks)   # ... and gone here
    rec, det, summary = hs.host_het_search(problem, space)
    ocl = orc.OracleCluster(os.path.join(root, 'hostfile'), os.path.join(root, 'clusterfile.json'), corrected=fix)
    oprof, _ = orc.load_profile_dir(os.path.join(root, 'profile'), meta['file_order'])
    omodel = orc.OracleModel(w.num_layers, w.hidden_size, w.sequence_length, w.vocab_size, oprof['model']['parameters'])
    want, counters = orc.het_search(oprof, ocl, omodel, seqs, w.gbs, w.num_layers, w.variance, w.max_permute_len,
                                    w.max_tp, w.max_bs, corrected=fix)
    assert (space.num_plans, summary.num_partition_calls, summary.num_records) == (counters['A'], counters['B'], counters['C'])
    got = hs.unpack_candidates(rec, det, space)
    assert len(got) == len(want)
    for g, x in zip(got, want):
        assert (g[0], g[1], g[3], g[4], g[5], g[6], g[7], g[8]) == (x[0], x[1], x[3], x[4], x[5], x[6], x[7], x[8])
    gold_costs = set(arr['cost'].tolist())
    assert any(x[8] not in gold_costs for x in want)                      # Q2 changes costs of multi-node stages


@pytest.mark.parametrize('name,fix,mode', [('mix32', ('Q5',), 0), ('mix32', ('Q5',), 2), ('c2_v100', ('Q6',), 1),
                                           ('c2_v100', ('Q5',), 2), ('mix32', ('Q6',), 2),
                                           ('mix32', ('Q1', 'Q2', 'Q5', 'Q6'), 1), ('c2_v100', ('Q1', 'Q2', 'Q5', 'Q6'), 0)])
def test_opt_in_corrected_mode_on_device(name, fix, mode, workload_dir):
    """SURVEY.md 8(f)-4, the device half: 'Q5' (no layer dropped by the vote) and 'Q6' (memory demand from the stage's
    own device type) change the evaluation itself (METIS_FIX_* bits of MetisProblem.corrected).  The device code, in
    every schedule, equals the oracle run with the same corrections bit for bit; with 'Q5' every partition ends at
    num_layers; the result differs from the strict search.  Never the default."""
    from oracle import metis_oracle as orc
    meta, arr = load_golden(name)
    w, root, _ = workload_dir(name)
    cluster, profile, _types, cfg = hs.load_inputs(root, 'profile', meta['file_order'], w.num_layers, w.hidden_size,
                                                   w.sequence_length, w.vocab_size)
    seqs = [tuple(s) for s in meta['node_sequences']]
    problem = flatten.build_problem(profile, cluster, cfg, w.gbs, w.max_tp, w.max_bs, seqs, corrected=fix)
    space = flatten.build_plan_space(len(seqs), cluster.get_total_num_devices(), w.gbs, w.num_layers, w.variance,
                                     w.max_permute_len, corrected=fix)
    rec, det, summary = hs.host_het_search(problem, space, mode=mode)
    ocl = orc.OracleCluster(os.path.join(root, 'hostfile'), os.path.join(root, 'clusterfile.json'), corrected=fix)
    oprof, _ = orc.load_profile_dir(os.path.join(root, 'profile'), meta['file_order'])
    omodel = orc.OracleModel(w.num_layers, w.hidden_size, w.sequence_length, w.vocab_size, oprof['model']['parameters'])
    want, counters = orc.het_search(oprof, ocl, omodel, seqs, w.gbs, w.num_layers, w.variance, w.max_permute_len,
                                    w.max_tp, w.max_bs, corrected=fix)
    assert (space.num_plans, summary.num_partition_calls, summary.num_balancer_runs, summary.num_records) == \
        (counters['A'], counters['B'], counters['runs'], counters['C'])
    got = hs.unpack_candidates(rec, det, space)
    assert len(got) == len(want)
    for g, x in zip(got, want):
        assert (g[0], g[1], g[3], g[4], g[5], g[6], g[7]) == (x[0], x[1], x[3], x[4], x[5], x[6], x[7])
        assert g[8] == x[8]
    if 'Q5' in fix:
        assert all(x[6][-1] == w.num_layers for x in want)                 # nothing dropped
    gold = {(int(o), int(st)): c for o, st, c in zip(arr['ordinal'], arr['step'], arr['cost'])}
    if set(fix) <= {'Q5', 'Q6'}:
        assert len(want) != len(gold) or any(gold.get((x[0], x[1])) != x[8] for x in want)   # not the strict result


def test_layer_balancer_random_vs_oracle_on_host():
    """The GPU suite's seeded balancer fuzz, on the host build of the device code: 1 600 random instances of
    LayerComputeBalancer.run (1-64 stages, 7-128 layers, capacities that over- and under-subscribe the layers)."""
    import random
    from oracle import metis_oracle as orc
    rng = random.Random(11)
    for L in (7, 24, 96, 128):
        lc = [0.01 + rng.random() for _ in range(L)]
        tot = sum(lc)
        lc = [x / tot for x in lc]
        rows = []
        for _ in range(400):
            S = rng.randint(1, min(L, 64))
            capa = [rng.random() ** rng.choice([1, 3]) + 1e-3 for _ in range(S)]
            t = sum(capa) * rng.choice([1.0, 1.0, 0.97, 1.05])
            rows.append([c / t for c in capa])
        got = hs.host_layer_balance(rows, lc, L)
        for capa, g in zip(rows, got):
            assert g == orc.layer_compute_balance(len(capa), L, list(capa), lc)


def test_random_homo_clusters_vs_oracle(tmp_path):
    """Seeded fuzz of the homogeneous path: HomoCostEstimator.get_cost of every UniformPlan of 60 random
    single-type clusters (device code, host build) against the oracle - plans kept, plans skipped by KeyError and
    every fp64 cost."""
    import random
    from oracle import metis_oracle as orc
    from metis_b200 import api
    from metis_b200.workloads import Workload, materialize, profile_file_order
    rng = random.Random(77)
    costed = skipped = 0
    for idx in range(60):
        dev = rng.choice(['A100', 'H100', 'B200', 'V100'])
        per = rng.choice([2, 4, 8])
        nn = rng.choice([1, 2, 4]) if per == 8 else rng.choice([1, 2, 3, 4])
        w = Workload(f'homo{idx}', [(dev, per)] * nn, rng.randint(6, 40), rng.choice([8, 16, 24, 32, 64, 96]),
                     rng.choice([1024, 4096]), rng.choice([512, 2048]), 51200, max_tp=rng.choice([1, 2, 4]),
                     tps=(1, 2, 4), bss=rng.choice([(1, 2, 4), (1, 2, 4, 8), (1, 2)]), seed=1000 + idx,
                     memory_gb={dev: rng.choice([8, 16, 40, 80])})
        root = str(tmp_path / w.name)
        materialize(w, root)
        order = profile_file_order(w)
        cluster, profile, types, cfg = hs.load_inputs(root, 'profile', order, w.num_layers, w.hidden_size,
                                                      w.sequence_length, w.vocab_size)
        plans = np.array([[p.dp, p.pp, p.tp, p.mbs, p.gbs]
                          for p in api.UniformPlanGenerator(cluster.get_total_num_devices(), w.max_tp, w.gbs)
                          if p.gbs == w.gbs], dtype=np.int32)
        if not len(plans):
            continue
        problem = flatten.build_problem(profile, cluster, cfg, w.gbs, int(plans[:, 2].max()), int(plans[:, 3].max()),
                                        [tuple(dict.fromkeys(t.name for t in cluster.get_device_types()))])
        cost, status = hs.host_homo_cost(problem, problem.type_names.index(types[0]), plans)
        ocl = orc.OracleCluster(os.path.join(root, 'hostfile'), os.path.join(root, 'clusterfile.json'))
        oprof, otypes = orc.load_profile_dir(os.path.join(root, 'profile'), order)
        omodel = orc.OracleModel(w.num_layers, w.hidden_size, w.sequence_length, w.vocab_size, oprof['model']['parameters'])
        want, counters = orc.homo_search(oprof, ocl, omodel, otypes[0], w.gbs, w.max_tp)
        keep = status != 1
        assert counters['matched'] == len(plans) and counters['keyerr'] == int((~keep).sum()), w
        assert plans[keep].tolist() == [list(p) for p, _ in want], w
        assert cost[keep].tolist() == [c for _, c in want], w
        costed += len(want)
        skipped += counters['keyerr']
    assert costed > 500 and skipped > 0, (costed, skipped)


@pytest.mark.parametrize('name', ['c1', 'mix32', 'c2_het16'])
def test_verbose_transcript_equals_the_reference(name, workload_dir):
    """SURVEY.md 8(f)-2: every line the reference prints while it searches (inter_stage_plan, invalid / valid
    strategies, stage performance, each partition attempt with its memory demand and state, re-weighted performance,
    'data loadbalancer', cost terms, cost / KeyError) - 499 / 10 201 / 32 796 lines captured from the unmodified
    reference (make_golden.py transcript:<name>) - against metis_b200.verbose.format_plan fed with the device's trace
    replay (metis_trace.cuh, here in its host build).  Byte for byte."""
    import ctypes as C
    import gzip
    from metis_b200 import api, verbose
    from metis_b200.arguments import parse_args
    from metis_b200.utils import DeviceType
    meta = json.load(open(os.path.join(GOLDEN, f'transcript_{name}.json')))
    gold = gzip.open(os.path.join(GOLDEN, f'transcript_{name}.txt.gz'), 'rt').read().split('\n')
    if name == 'c1':
        root, sub = C1_DIR, 'profile_data_samples'
        argv = ['--num_layers', '10', '--gbs', '128', '--max_profiled_tp_degree', '4', '--max_profiled_batch_size', '4',
                '--min_group_scale_variance', '1', '--max_permute_len', '4', '--hidden_size', '4096',
                '--sequence_length', '1024', '--vocab_size', '51200', '--attention_head_size', '32']
    else:
        w, root, digest = workload_dir(name)
        assert digest == meta['inputs_sha256']
        sub, argv = 'profile', w.cli_args(root)
    args = parse_args(argv)
    cluster, profile, _types, cfg = hs.load_inputs(root, sub, meta['file_order'], args.num_layers, args.hidden_size,
                                                   args.sequence_length, args.vocab_size)
    seqs = [tuple(DeviceType[t] for t in seq) for seq in meta['node_sequences']]
    problem, space, _ = api.het_problem(args, cluster, profile, cfg, None, seqs)
    keep = dict(problem.arrays)
    keep.update(blocks=space.blocks, batches=space.batches, rows=space.rows)
    p = problem.as_struct(lambda n: keep[n].ctypes.data)
    sp = space.as_struct(lambda n: keep[n].ctypes.data)
    n, words = space.num_plans, max(256, 64 * (4 * sp.max_stage + 24))
    ords = np.arange(n, dtype=np.uint32)
    trace = np.zeros((n, words), dtype=np.uint64)
    hs.hostsim().hostsim_het_trace(C.byref(p), C.byref(sp), C.c_void_p(ords.ctypes.data), C.c_int64(n),
                                   C.c_void_p(trace.ctypes.data), C.c_int32(words))
    lines = []
    for o in range(n):
        ns, label, row, batches, codes = space.locate(o)
        plan = api.InterStagePlan(ns_idx=ns, node_sequence=seqs[ns], dg_idx=row, device_groups=[1 << int(c) for c in codes],
                                  num_stage=label, batches=batches, gbs=args.gbs)
        lines += list(verbose.format_plan(trace[o], plan, cluster, args.max_profiled_tp_degree, args.max_profiled_batch_size))
    end = next(i for i, l in enumerate(gold) if l.startswith('search_time:'))
    assert len(lines) == end - 1
    assert lines == gold[1:end]


@pytest.mark.parametrize('name', ['mix32', 'c2_het16'])
def test_lazy_result_object_on_host_records(name, workload_dir):
    """Host logic of the drop-in API without a GPU: records / detail rows of the host build go through
    search.Candidates and api.HetSearchResult (the objects cost_het_cluster() returns) - length, indexing, slices,
    iteration, ranked() (Python's stable sort when no device permutation is given), best() by bisection on the
    kernels' argmin key - and must give the golden 7-tuples."""
    from metis_b200 import api, search
    meta, arr = load_golden(name)
    w, root, _ = workload_dir(name)
    cluster, profile, _types, cfg = hs.load_inputs(root, 'profile', meta['file_order'], w.num_layers, w.hidden_size,
                                                   w.sequence_length, w.vocab_size)
    seqs = [tuple(s) for s in meta['node_sequences']]
    problem = flatten.build_problem(profile, cluster, cfg, w.gbs, w.max_tp, w.max_bs, seqs)
    space = flatten.build_plan_space(len(seqs), cluster.get_total_num_devices(), w.gbs, w.num_layers, w.variance,
                                     w.max_permute_len)
    rec, det, summary = hs.host_het_search(problem, space, mode=1)
    order = np.lexsort((rec['step'], rec['ordinal']))              # estimate_costs order, like metis_sort_records
    rec, det = rec[order], det[order]
    cand = search.Candidates(rec, det, space, seqs)
    best = (int(summary.best.ordinal), int(summary.best.step))
    res = api.HetSearchResult(cand, None, {}, best_key=best)
    gold = [(tuple(meta['node_sequences'][g[2]]), g[3], g[4], g[5], g[6], g[7], g[8]) for g in golden_rows(arr)]
    assert len(res) == len(gold) and list(res) == gold and res == gold
    assert res[0] == gold[0] and res[-1] == gold[-1] and res[3:7] == gold[3:7]
    with pytest.raises(IndexError):
        res[len(gold)]
    want = sorted(gold, key=lambda kv: kv[6])
    assert res.best() == want[0]                                   # before any ranking exists: bisection
    assert res.rank_order is None
    assert res.ranked(5) == want[:5] and res.ranked() == want      # stable sort fallback
    assert res.best() == want[0]
    assert (res.costs == np.array([g[6] for g in gold])).all()
    # a device-rows space (rows only on the GPU) falls back to the host enumerator when asked on the host
    lazy_space = flatten.build_plan_space(len(seqs), cluster.get_total_num_devices(), w.gbs, w.num_layers, w.variance,
                                          w.max_permute_len, device_rows=True)
    assert list(api.HetSearchResult(search.Candidates(rec, det, lazy_space, seqs), None, {})) == gold
