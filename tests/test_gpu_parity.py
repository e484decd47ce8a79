"""GPU parity tests (run with -m gpu on the B200 box).  Everything goes through the C ABI of
libmetis_b200.so via ctypes (metis_b200.native / metis_b200.search) and is compared bit-for-bit
with (a) golden files produced by the unmodified reference and (b) the CPU oracle on the same
seeded inputs.  Integer outputs (partitions, strategies, ordinals, counters) and fp64 costs must be
identical - the tolerance north_star allows for costs (1e-6 relative) is not used.
"""
import gzip
import itertools
import json
import os
import random

import numpy as np
import pytest

from conftest import C1_DIR, GOLDEN, assert_candidates_equal, device_columns, golden_best, golden_rows, load_golden
from golden_units import load_units

pytestmark = pytest.mark.gpu


def _gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from metis_b200 import native
    native.load_library()          # raises (test error, not skip) when the extension is missing
    return torch


def _inputs(root, profile_sub, file_order, num_layers, hidden, seq, vocab):
    from metis_b200.data_loader import ProfileDataLoader
    from metis_b200.gpu_cluster import GPUCluster
    from metis_b200.utils import ModelConfig
    cluster = GPUCluster(os.path.join(root, 'hostfile'), os.path.join(root, 'clusterfile.json'))
    profile, types = ProfileDataLoader(os.path.join(root, profile_sub), file_order).load_profile_data_all()
    cfg = ModelConfig(model_name='t', num_layers=num_layers, sequence_length=seq, vocab_size=vocab,
                      hidden_size=hidden, attention_head_size=32)
    return cluster, profile, types, cfg


def _device_search(meta, root, profile_sub, w, rank=0, world=1, tile=128, want_detail=True):
    from metis_b200 import flatten, search
    cluster, profile, _, cfg = _inputs(root, profile_sub, meta['file_order'], w['L'], w['hidden'], w['seq'], w['vocab'])
    seqs = [tuple(s) for s in meta['node_sequences']]
    problem = flatten.build_problem(profile, cluster, cfg, w['gbs'], w['max_tp'], w['max_bs'], seqs)
    space = flatten.build_plan_space(len(seqs), cluster.get_total_num_devices(), w['gbs'], w['L'], w['variance'],
                                     w['mpl'])
    dp = search.DeviceProblem(problem, space, 'cuda:0')
    out = search.HetSearcher(dp, rank, world, tile, want_records=True, want_detail=want_detail).run()
    return problem, space, out


def _cfg(w):
    return dict(L=w.num_layers, hidden=w.hidden_size, seq=w.sequence_length, vocab=w.vocab_size, gbs=w.gbs,
                variance=w.variance, mpl=w.max_permute_len, max_tp=w.max_tp, max_bs=w.max_bs)


def _assert_arrays_equal(out, space, arr, meta):
    """Vectorised comparison of sorted device records with the golden (conftest.assert_candidates_equal)."""
    assert_candidates_equal(device_columns(out.records, out.detail, arr['dp'].shape[1]), meta, arr)


def test_c1_het_and_homo_vs_golden_and_oracle():
    _gpu()
    from metis_b200 import api, search
    from oracle import metis_oracle as orc
    meta, arr = load_golden('c1_het')
    w = dict(L=10, hidden=4096, seq=1024, vocab=51200, gbs=128, variance=1, mpl=4, max_tp=4, max_bs=4)
    problem, space, out = _device_search(meta, C1_DIR, 'profile_data_samples', w)
    assert space.num_plans == 32 and out.summary['num_records'] == 19
    assert out.summary['num_partition_calls'] == meta['counters']['B']
    _assert_arrays_equal(out, space, arr, meta)
    assert out.best[:3] == (621.8881853975784, 7, 0)
    # same inputs through the oracle (not the golden file)
    ocl = orc.OracleCluster(os.path.join(C1_DIR, 'hostfile'), os.path.join(C1_DIR, 'clusterfile.json'))
    oprof, otypes = orc.load_profile_dir(os.path.join(C1_DIR, 'profile_data_samples'), meta['file_order'])
    omodel = orc.OracleModel(10, 4096, 1024, 51200, oprof['model']['parameters'])
    want, _ = orc.het_search(oprof, ocl, omodel, [tuple(s) for s in meta['node_sequences']], 128, 10, 1, 4, 4, 4)
    got = search.materialize(out.records, out.detail, space, [tuple(s) for s in meta['node_sequences']])
    assert [(g[1], g[2], g[3], g[4], g[5], g[6]) for g in got] == [(x[3], x[4], x[5], x[6], x[7], x[8]) for x in want]
    # homo path (KAT-2)
    hmeta, harr = load_golden('c1_homo')
    cluster, profile, types, cfg = _inputs(C1_DIR, 'profile_data_samples', hmeta['file_order'], 10, 4096, 1024, 51200)
    from metis_b200.arguments import parse_args
    args = parse_args(['--gbs', '128', '--max_profiled_tp_degree', '4', '--num_layers', '10'])
    volume = api.GPTActivationAndParam(cfg, profile['model']['parameters'])
    hom = api.cost_homo_cluster(args, cluster, api.HomoCostEstimator(profile, cfg, volume, cluster), types[0], 'cuda:0')
    assert [[p.dp, p.pp, p.tp, p.mbs, p.gbs] for p, _ in hom] == harr['plan'].tolist()
    assert [c for _, c in hom] == harr['cost'].tolist()
    assert min(c for _, c in hom) == 621.8881853975784


@pytest.mark.parametrize('name', ['c2_het16', 'c2_v100', 'mix32', 'het32_tight', 'sweep_n8_t1', 'sweep_n16_t2_v0',
                                  'sweep_n32_t4', 'long_profile', 'q10_big_first'])
def test_synthetic_vs_golden(name, workload_dir):
    _gpu()
    meta, arr = load_golden(name)
    w, root, digest = workload_dir(name)
    assert digest == meta['inputs_sha256']
    problem, space, out = _device_search(meta, root, 'profile', _cfg(w))
    c = meta['counters']
    assert space.num_plans == c['A']
    s = out.summary
    assert (s['num_partition_calls'], s['num_balancer_runs'], s['num_records'], s['num_keyerror']) == \
        (c['B'], c['runs'], c['C'], c['keyerr'])
    assert s['fatal_ordinal'] == 2 ** 64 - 1
    _assert_arrays_equal(out, space, arr, meta)
    gold = golden_rows(arr)
    best = min(gold, key=lambda g: (g[8], g[0], g[1]))
    assert out.best[:3] == (best[8], best[0], best[1])


@pytest.mark.parametrize('name', ['c3_homo64_mpl4', 'c3_homo64_mpl6'])
def test_full_size_c3_vs_golden(name, workload_dir):
    """BASELINE configs[2] at full size (8.3e4 / 7.7e5 inter-stage plans): every costed candidate."""
    _gpu()
    meta, arr = load_golden(name)
    w, root, digest = workload_dir(name)
    assert digest == meta['inputs_sha256']
    problem, space, out = _device_search(meta, root, 'profile', _cfg(w))
    c = meta['counters']
    assert space.num_plans == c['A']
    s = out.summary
    assert (s['num_partition_calls'], s['num_balancer_runs'], s['num_records']) == (c['B'], c['runs'], c['C'])
    _assert_arrays_equal(out, space, arr, meta)
    assert out.best[:3] == golden_best(meta, arr)


@pytest.mark.parametrize('env', [{'METIS_CHAIN_THREADS': '64'}, {'METIS_SMEM_BLOB_MAX': '0'},
                                 {'METIS_CHAIN_THREADS': '128', 'METIS_SMEM_BLOB_MAX': '0'}, {'METIS_SAVE_SLOTS': '40'}],
                         ids=['chain_blocks_of_2_warps', 'tables_in_global_memory', 'both', 'hand_over_store_full'])
def test_launch_shapes_give_the_same_records(env, workload_dir, monkeypatch):
    """Other block shapes of the chain kernel, tables left in global memory (instead of the TMA-staged shared copy)
    and a hand-over store with room for 40 continuations only (the others replay their first attempt) must still
    produce every golden candidate of the 8.3e4-plan space."""
    _gpu()
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    meta, arr = load_golden('c3_homo64_mpl4')
    w, root, _ = workload_dir('c3_homo64_mpl4')
    problem, space, out = _device_search(meta, root, 'profile', _cfg(w))
    c = meta['counters']
    s = out.summary
    assert (s['num_partition_calls'], s['num_balancer_runs'], s['num_records']) == (c['B'], c['runs'], c['C'])
    _assert_arrays_equal(out, space, arr, meta)


@pytest.mark.parametrize('name', ['c4_het128', 'c4_het128_mpl6', 'sweep_n128_t1_v0', 'sweep_n256_t2_v0'])
def test_sampled_vs_golden(name, workload_dir):
    """Spaces too large for the reference to finish: BASELINE configs[3] (3 types, 128 GPUs: 4.5e6 plans, and 6.8e7
    with max_permute_len 6) and two variance-0 points of configs[4] at 128 / 256 GPUs.  The reference was run on a
    STRATIFIED sample of the ordinals - the first two, the middle and the last device-group row of EVERY
    (node sequence, stage count) block with every divisor of gbs (this covers every mislabelled Q1 block) plus a
    uniform share of all ordinals (make_golden.py name:strat).  The GPU searches the whole space; every sampled
    candidate must match (counters per sample included), and the summary's best must be the argmin of all records."""
    _gpu()
    from metis_b200 import flatten, search
    meta, arr = load_golden(name)
    w, root, digest = workload_dir(name)
    assert digest == meta['inputs_sha256']
    cfg = _cfg(w)
    cluster, profile, _, mc = _inputs(root, 'profile', meta['file_order'], cfg['L'], cfg['hidden'], cfg['seq'], cfg['vocab'])
    seqs = [tuple(s) for s in meta['node_sequences']]
    problem = flatten.build_problem(profile, cluster, mc, cfg['gbs'], cfg['max_tp'], cfg['max_bs'], seqs)
    space = flatten.build_plan_space(len(seqs), cluster.get_total_num_devices(), cfg['gbs'], cfg['L'], cfg['variance'], cfg['mpl'])
    assert space.num_plans == meta['counters']['A']
    searcher = search.HetSearcher(search.DeviceProblem(problem, space, 'cuda:0'), want_records=True, want_detail=False)
    out = searcher.run()
    assert out.summary['fatal_ordinal'] == 2 ** 64 - 1
    rec = out.records
    keep = np.isin(rec['ordinal'].astype(np.int64), arr['sample'])
    sub = rec[keep]
    assert len(sub) == meta['counters']['C']
    stride = 3 * int(space.blocks['num_stage'].max()) + 1

    class Sub:
        records = sub
        detail = searcher.detail_for(sub)[:, :max(stride, arr['dp'].shape[1] * 3 + 1)]
    _assert_arrays_equal(Sub, space, arr, meta)
    # every block of the space has sampled plans, and the blocks with costed candidates appear in the comparison
    blk_of = np.searchsorted(space.blocks['first_ordinal'], arr['sample'], side='right') - 1
    assert len(np.unique(blk_of)) == len(space.blocks)
    # checksum-style property at full size: the summary's best is the argmin of all records
    i = int(np.lexsort((rec['step'], rec['ordinal'], rec['cost']))[0])
    assert out.best[:3] == (float(rec['cost'][i]), int(rec['ordinal'][i]), int(rec['step'][i]))


@pytest.mark.parametrize('name', ['c3_homo64_mpl4', 'sweep_n8_t1'])
def test_homo_synthetic_vs_golden(name, workload_dir):
    _gpu()
    from metis_b200 import api
    from metis_b200.arguments import parse_args
    meta, arr = load_golden(name + '_homo')
    w, root, digest = workload_dir(name)
    assert digest == meta['inputs_sha256']
    cluster, profile, types, cfg = _inputs(root, 'profile', meta['file_order'], w.num_layers, w.hidden_size,
                                           w.sequence_length, w.vocab_size)
    args = parse_args(['--gbs', str(w.gbs), '--max_profiled_tp_degree', str(w.max_tp), '--num_layers', str(w.num_layers)])
    volume = api.GPTActivationAndParam(cfg, profile['model']['parameters'])
    hom = api.cost_homo_cluster(args, cluster, api.HomoCostEstimator(profile, cfg, volume, cluster), types[0], 'cuda:0')
    assert [[p.dp, p.pp, p.tp, p.mbs, p.gbs] for p, _ in hom] == arr['plan'].tolist()
    assert [c for _, c in hom] == arr['cost'].tolist()


def test_fatal_keyerror_like_reference(workload_dir):
    _gpu()
    from metis_b200 import search
    meta, _ = load_golden('fatal_gbs96')
    w, root, _ = workload_dir('fatal_gbs96')
    problem, space, out = _device_search(meta, root, 'profile', _cfg(w))
    assert out.summary['fatal_ordinal'] == meta['fatal'][0]
    with pytest.raises(KeyError) as err:
        search.raise_fatal(out.summary, problem)
    assert str(err.value) == meta['fatal'][2]


@pytest.mark.parametrize('name', ['q10_small_first', 'q10_small_first_t1'])
def test_fatal_indexerror_unequal_nodes(name, workload_dir):
    """Nodes with different GPU counts, node 0 the smallest (quirk Q10, gpu_cluster.py:25-26 + load_balancer.py:109-119):
    the reference dies with IndexError; so does the drop-in, at the same plan."""
    _gpu()
    from metis_b200 import search
    meta, _ = load_golden(name)
    w, root, _ = workload_dir(name)
    problem, space, out = _device_search(meta, root, 'profile', _cfg(w))
    assert out.summary['fatal_ordinal'] == meta['fatal'][0]
    with pytest.raises(IndexError) as err:
        search.raise_fatal(out.summary, problem)
    assert str(err.value) == meta['fatal'][2]


def test_shards_partition_the_space(workload_dir):
    """Multi-GPU sharding property on one device: the union of the shards' records is the whole
    search, and the lexicographic min of the shard bests is the global best."""
    _gpu()
    meta, arr = load_golden('c3_homo64_mpl4')
    w, root, _ = workload_dir('c3_homo64_mpl4')
    recs, bests, counters = [], [], np.zeros(3, dtype=np.int64)
    for rank in range(4):
        _, space, out = _device_search(meta, root, 'profile', _cfg(w), rank=rank, world=4, tile=256, want_detail=False)
        recs.append(out.records)
        bests.append(out.best)
        counters += [out.summary['num_partition_calls'], out.summary['num_balancer_runs'], out.summary['num_records']]
    rec = np.concatenate(recs)
    rec = rec[np.lexsort((rec['step'], rec['ordinal']))]
    assert (rec['ordinal'].astype(np.int64) == arr['ordinal']).all()
    assert (rec['cost'].view(np.uint64) == arr['cost'].view(np.uint64)).all()
    c = meta['counters']
    assert counters.tolist() == [c['B'], c['runs'], c['C']]
    i = int(np.lexsort((arr['step'], arr['ordinal'], arr['cost']))[0])
    assert min(b[:3] for b in bests if b) == (float(arr['cost'][i]), int(arr['ordinal'][i]), int(arr['step'][i]))


def test_rerun_is_idempotent(workload_dir):
    _gpu()
    from metis_b200 import flatten, search
    meta, _ = load_golden('c2_v100')
    w, root, _ = workload_dir('c2_v100')
    cfg = _cfg(w)
    cluster, profile, _, mc = _inputs(root, 'profile', meta['file_order'], cfg['L'], cfg['hidden'], cfg['seq'], cfg['vocab'])
    seqs = [tuple(s) for s in meta['node_sequences']]
    problem = flatten.build_problem(profile, cluster, mc, w.gbs, w.max_tp, w.max_bs, seqs)
    space = flatten.build_plan_space(len(seqs), 16, w.gbs, w.num_layers, w.variance, w.max_permute_len)
    searcher = search.HetSearcher(search.DeviceProblem(problem, space, 'cuda:0'), want_detail=True, capacity=8)
    a = searcher.run()            # capacity 8 forces the grow-and-rerun path
    b = searcher.run()
    assert a.summary == b.summary and a.best == b.best
    assert (a.records == b.records).all()
    for i in range(len(a.records)):               # bytes past 3S+1 of a detail row are unspecified
        S = int(a.records['num_stage'][i])
        assert (a.detail[i, :3 * S + 1] == b.detail[i, :3 * S + 1]).all()
    picks = a.records[[0, len(a.records) // 2, len(a.records) - 1]]
    replay = searcher.detail_for(picks)
    for k, i in enumerate([0, len(a.records) // 2, len(a.records) - 1]):
        S = int(a.records['num_stage'][i])
        assert (replay[k, :3 * S + 1] == a.detail[i, :3 * S + 1]).all()


def test_layer_balancer_units_on_gpu():
    _gpu()
    from metis_b200 import search
    units = load_units()
    by_l = {}
    for case in units['balancer']:
        by_l.setdefault((case['L'], tuple(case['lc'])), []).append(case)
    for (L, lc_hex), cases in by_l.items():
        lc = [float.fromhex(x) for x in lc_hex]
        got = search.layer_balance([[float.fromhex(x) for x in c['capa']] for c in cases], lc, L, 'cuda:0')
        for g, c in zip(got, cases):
            assert g == c['part'], c


def test_layer_balancer_random_vs_oracle():
    """Seeded random instances straight against the oracle's list-based restatement."""
    _gpu()
    from metis_b200 import search
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
        got = search.layer_balance(rows, lc, L, 'cuda:0')
        for capa, g in zip(rows, got):
            assert g == orc.layer_compute_balance(len(capa), L, list(capa), lc)


def test_cli_transcript_matches_reference_format(capsys):
    """cost_het_cluster.py drop-in CLI on the README example: ranked table identical to KAT-1."""
    _gpu()
    import cost_het_cluster as cli
    order_first = 'DeviceType.A100_tp2_bs2.json'
    meta, arr = load_golden('c1_het')
    # the CLI uses os.listdir order; pin it by pointing the loader at a copy listed in golden order
    import shutil
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        # os.listdir order is filesystem dependent: copy files one by one in the golden order and
        # fall back to comparing only order-independent facts if the filesystem re-orders them
        dst = os.path.join(tmp, 'p')
        os.makedirs(dst)
        for f in meta['file_order']:
            shutil.copy(os.path.join(C1_DIR, 'profile_data_samples', f), dst)
        listed = [f for f in os.listdir(dst) if f.endswith('.json')]
        ranked = cli.main(['--model_name', 'GPT', '--model_size', '1.5B', '--num_layers', '10', '--gbs', '128',
                           '--hostfile_path', os.path.join(C1_DIR, 'hostfile'),
                           '--clusterfile_path', os.path.join(C1_DIR, 'clusterfile.json'),
                           '--profile_data_path', dst, '--max_profiled_tp_degree', '4',
                           '--max_profiled_batch_size', '4', '--min_group_scale_variance', '1',
                           '--max_permute_len', '4', '--hidden_size', '4096', '--sequence_length', '1024',
                           '--vocab_size', '51200', '--attention_head_size', '32'])
    text = capsys.readouterr().out
    assert 'len(costs): 19' in text
    assert 'rank, cost, node_sequence, device_groups, strategies(dp_deg, tp_deg), batches(number of batch), layer_partition' in text
    assert len(ranked) == 19
    if listed[0] == order_first:
        assert "1, 621.8881853975784, (<DeviceType.A100: 'a100'>,), [64], [(64, 1)], 1, [0, 10]" in text


def _sort_on_device(rec_np, mode):
    import ctypes as C
    import torch
    from metis_b200 import native
    lib = native.load_library()
    n = len(rec_np)
    raw = torch.from_numpy(rec_np.view(np.uint8).reshape(-1).copy()).cuda() if n else torch.zeros(16, dtype=torch.uint8).cuda()
    perm = torch.full((max(n, 1),), -1, dtype=torch.int32, device='cuda')
    ws = torch.empty(int(lib.metis_sort_workspace_bytes(n)), dtype=torch.uint8, device='cuda')
    rc = lib.metis_sort_records(C.c_void_p(raw.data_ptr()), C.c_int64(n), C.c_int32(mode), C.c_void_p(perm.data_ptr()),
                                C.c_void_p(ws.data_ptr()), C.c_int64(ws.numel()),
                                C.c_void_p(torch.cuda.current_stream().cuda_stream))
    native.check(rc, 'metis_sort_records')
    torch.cuda.synchronize()
    out = raw.cpu().numpy()[:n * 16].view(native.RECORD_DTYPE) if n else rec_np[:0]
    return out, perm.cpu().numpy()[:n].view(np.uint32)


@pytest.mark.parametrize('n', [0, 1, 31, 32, 33, 1000, 100003, 300000])
def test_record_sort_is_the_stable_python_sort(n):
    """metis_sort_records against numpy's stable sorts: many equal costs (ties must keep estimate_costs
    order, cost_het_cluster.py:76), negative / huge / infinite costs, ordinals up to 2^32, steps up to 2^16."""
    _gpu()
    from metis_b200 import native
    rng = np.random.default_rng(n + 5)
    rec = np.zeros(n, dtype=native.RECORD_DTYPE)
    pool = np.concatenate([rng.uniform(-1e3, 1e6, 40), [np.inf, 1e300, 5e-324, 1.0, 1.0000000000000002, -7.5]])
    rec['cost'] = rng.choice(pool, n)
    rec['ordinal'] = rng.integers(0, 2 ** 32 - 32, n, dtype=np.uint64).astype(np.uint32) if n % 2 else rng.integers(0, 5000, n)
    rec['step'] = rng.integers(0, 2 ** 16, n) if n % 3 == 0 else rng.integers(0, 19, n)
    rec['num_repartition'] = rng.integers(1, 4, n)
    rec['num_stage'] = rng.integers(1, 129, n)
    got, perm = _sort_on_device(rec, native.SORT_POSITION)
    want = np.lexsort((rec['step'], rec['ordinal']))
    assert (perm == want).all() and (got.view(np.uint8) == rec[want].view(np.uint8)).all()
    got, perm = _sort_on_device(rec, native.SORT_RANKED)
    want = np.lexsort((rec['step'], rec['ordinal'], rec['cost']))
    assert (perm == want).all() and (got.view(np.uint8) == rec[want].view(np.uint8)).all()
    got, perm = _sort_on_device(rec, native.SORT_BY_COST_STABLE)
    want = np.argsort(rec['cost'], kind='stable')
    assert (perm == want).all() and (got.view(np.uint8) == rec[want].view(np.uint8)).all()


def test_ranked_listing_is_sorted_estimate_costs(workload_dir):
    """The ranked list of the CLI (cost_het_cluster.py:76-80) from the device sort equals Python's
    sorted(estimate_costs, key=cost) on the golden candidates of the reference."""
    torch = _gpu()
    from metis_b200 import flatten, search
    meta, arr = load_golden('c3_homo64_mpl4')
    w, root, _ = workload_dir('c3_homo64_mpl4')
    cfg = _cfg(w)
    cluster, profile, _, mc = _inputs(root, 'profile', meta['file_order'], cfg['L'], cfg['hidden'], cfg['seq'], cfg['vocab'])
    seqs = [tuple(s) for s in meta['node_sequences']]
    problem = flatten.build_problem(profile, cluster, mc, cfg['gbs'], cfg['max_tp'], cfg['max_bs'], seqs)
    space = flatten.build_plan_space(len(seqs), cluster.get_total_num_devices(), cfg['gbs'], cfg['L'], cfg['variance'], cfg['mpl'])
    out = search.HetSearcher(search.DeviceProblem(problem, space, 'cuda:0'), want_records=True, want_ranking=True).run()
    gold_cost = arr['cost']
    want = sorted(range(len(gold_cost)), key=lambda i: gold_cost[i])         # Python's stable sort, as the reference
    assert out.rank_order.tolist() == want
    assert (out.records['cost'].view(np.uint64) == gold_cost.view(np.uint64)).all()


@pytest.mark.parametrize('name', ['mix32', 'het32_tight', 'c2_het16', 'c3_homo64_mpl4'])
@pytest.mark.parametrize('factor', [1, 2 ** 31 - 1], ids=['bulk_round_then_chains', 'chain_kernel_only'])
def test_scheduler_modes_agree(name, factor, workload_dir):
    """The two schedules of a search are forced in turn (MetisShard.reserved): the bulk round (first partition
    attempt of every plan, one plan per thread) followed by the chain kernel for the plans that ran out of memory,
    and the chain kernel alone (one warp per plan from the first attempt on).  Both must reproduce every golden
    candidate, including the re-partition counts of mixed-type and memory-tight plans."""
    _gpu()
    from metis_b200 import flatten, search
    meta, arr = load_golden(name)
    w, root, _ = workload_dir(name)
    cfg = _cfg(w)
    cluster, profile, _, mc = _inputs(root, 'profile', meta['file_order'], cfg['L'], cfg['hidden'], cfg['seq'], cfg['vocab'])
    seqs = [tuple(s) for s in meta['node_sequences']]
    problem = flatten.build_problem(profile, cluster, mc, cfg['gbs'], cfg['max_tp'], cfg['max_bs'], seqs)
    space = flatten.build_plan_space(len(seqs), cluster.get_total_num_devices(), cfg['gbs'], cfg['L'], cfg['variance'], cfg['mpl'])
    s = search.HetSearcher(search.DeviceProblem(problem, space, 'cuda:0'), want_records=True, want_detail=True)
    s.shard.reserved = factor
    out = s.run()
    c = meta['counters']
    assert (out.summary['num_partition_calls'], out.summary['num_balancer_runs'], out.summary['num_records']) == \
        (c['B'], c['runs'], c['C'])
    _assert_arrays_equal(out, space, arr, meta)


def _api_inputs(name, workload_dir):
    from metis_b200 import api
    from metis_b200.arguments import parse_args
    meta, arr = load_golden(name)
    w, root, _ = workload_dir(name)
    args = parse_args(w.cli_args(root))
    cluster, profile, _types, cfg = _inputs(root, 'profile', meta['file_order'], w.num_layers, w.hidden_size,
                                            w.sequence_length, w.vocab_size)
    volume = api.GPTActivationAndParam(cfg, profile['model']['parameters'])
    est = api.HeteroCostEstimator(profile, cfg, volume, cluster)
    llb = api.LayerLoadBalancer(cluster, profile, cfg, args.gbs)
    seqs = [tuple(s) for s in meta['node_sequences']]
    return meta, arr, (args, cluster, profile, cfg, est, llb), seqs


def test_api_lazy_result_equals_eager_tuples(workload_dir):
    """api.cost_het_cluster (the function the reference's callers use, cost_het_cluster.py:71-74) on c3_homo64_mpl4:
    the lazy sequence equals the eagerly materialised 7-tuples and the golden candidates; ranked() is Python's
    stable sorted(); repeated calls reuse the cached engine and give the same answer."""
    _gpu()
    import time
    from metis_b200 import api, search
    meta, arr, call, seqs = _api_inputs('c3_homo64_mpl4', workload_dir)
    res = api.cost_het_cluster(*call, node_sequences=seqs, device='cuda:0')
    assert len(res) == meta['counters']['C'] == len(arr['cost'])
    assert (res.costs.view(np.uint64) == arr['cost'].view(np.uint64)).all()
    gold = golden_rows(arr)
    eager = search.materialize(res.candidates.records, res.candidates.detail_rows(np.arange(len(res))),
                               res.candidates.space, seqs)
    assert len(eager) == len(gold)
    for e, g in zip(eager, gold):
        assert (e[1], e[2], e[3], e[4], e[5], e[6]) == (g[3], g[4], g[5], g[6], g[7], g[8])
    assert res[0] == eager[0] and res[-1] == eager[-1] and res[1234] == eager[1234]
    assert res[10:13] == eager[10:13]
    lazy_all = list(res)
    assert lazy_all == eager and res == eager
    want_rank = sorted(eager, key=lambda kv: kv[6])
    assert res.ranked(25) == want_rank[:25]
    assert res.best() == want_rank[0]
    t0 = time.perf_counter()
    again = api.cost_het_cluster(*call, node_sequences=seqs, device='cuda:0')
    wall = time.perf_counter() - t0
    assert again.best() == want_rank[0] and len(again) == len(res)
    assert (again.costs.view(np.uint64) == res.costs.view(np.uint64)).all()
    assert wall < 2.0, f'second api.cost_het_cluster call took {wall:.3f} s'


def test_api_small_and_mixed_vs_golden(workload_dir):
    """The same through the cached engine for problems of different shapes back to back (buffers are re-used /
    re-grown): mixed-type stages, tight memory, 4 types."""
    _gpu()
    from metis_b200 import api
    for name in ('mix32', 'het32_tight', 'c2_het16', 'sweep_n32_t4', 'mix32'):
        meta, arr, call, seqs = _api_inputs(name, workload_dir)
        res = api.cost_het_cluster(*call, node_sequences=seqs, device='cuda:0')
        gold = golden_rows(arr)
        assert len(res) == len(gold), name
        got = list(res)
        for e, g in zip(got, gold):
            assert e == (tuple(meta['node_sequences'][g[2]]), g[3], g[4], g[5], g[6], g[7], g[8]), name
        assert res.ranked() == sorted(got, key=lambda kv: kv[6]), name


def test_c4_whole_space_vs_oracle_on_host_cores(workload_dir):
    """BASELINE configs[3] - the configuration north_star shards over 8 GPUs - compared in FULL: the pinned CPU oracle
    evaluates every one of the 4.5e6 inter-stage plans on this box's host cores (tests/oracle_pool.py, block-parallel)
    and every candidate it costs must equal the device's record - ordinal, chain step, strategies, layer partition,
    num_repartition and all 64 bits of the cost - and the device must not have any record the oracle lacks.
    METIS_ORACLE_BUDGET_S (default 900) bounds the oracle's wall time on a slow host: then at least a quarter of the
    space must have been compared and the coverage is reported in the assertion message / stdout."""
    _gpu()
    import oracle_pool
    from metis_b200 import flatten, search
    name = 'c4_het128'
    meta, _arr = load_golden(name)
    w, root, _ = workload_dir(name)
    cfg = _cfg(w)
    cluster, profile, _, mc = _inputs(root, 'profile', meta['file_order'], cfg['L'], cfg['hidden'], cfg['seq'], cfg['vocab'])
    seqs = [tuple(s) for s in meta['node_sequences']]
    problem = flatten.build_problem(profile, cluster, mc, cfg['gbs'], cfg['max_tp'], cfg['max_bs'], seqs)
    space = flatten.build_plan_space(len(seqs), cluster.get_total_num_devices(), cfg['gbs'], cfg['L'], cfg['variance'], cfg['mpl'])
    stride = 3 * int(space.blocks['num_stage'].max()) + 1
    out = search.HetSearcher(search.DeviceProblem(problem, space, 'cuda:0'), want_records=True, want_detail=True,
                             detail_stride=stride).run()
    assert out.summary['fatal_ordinal'] == 2 ** 64 - 1
    rec, det = out.records, out.detail
    key = (rec['ordinal'].astype(np.int64) << 16) | rec['step'].astype(np.int64)      # sorted: estimate_costs order
    seen = np.zeros(len(rec), dtype=bool)
    items = oracle_pool.work_items(space)
    budget = float(os.environ.get('METIS_ORACLE_BUDGET_S', '900'))
    done = plans = cands = 0
    totals = {'B': 0, 'runs': 0, 'keyerr': 0}
    ndiv = len(space.batches)
    for item, pk, counters in oracle_pool.run(root, name, meta['file_order'], seqs, items, budget):
        first, _ns, _label, stages, row_lo, row_hi = item
        lo_ord, hi_ord = first + row_lo * ndiv, first + row_hi * ndiv
        a, b = np.searchsorted(key, [lo_ord << 16, hi_ord << 16])
        n = len(pk['cost'])
        assert b - a == n, f'plans {lo_ord}..{hi_ord}: device has {b - a} candidates, oracle {n}'
        if n:
            r, d = rec[a:b], det[a:b]
            assert ((r['ordinal'].astype(np.int64) == pk['ordinal']) & (r['step'].astype(np.int64) == pk['step'])).all()
            assert (r['num_repartition'].astype(np.int64) == pk['nrep']).all()
            assert (r['cost'].view(np.uint64) == pk['cost'].view(np.uint64)).all(), f'cost bits differ in {lo_ord}..{hi_ord}'
            assert (r['num_stage'] == stages).all()
            assert ((1 << d[:, :stages].astype(np.int64)) == pk['dp']).all()
            assert ((1 << d[:, stages:2 * stages].astype(np.int64)) == pk['tp']).all()
            assert (d[:, 2 * stages:3 * stages + 1].astype(np.int64) == pk['part']).all()
            seen[a:b] = True
        done += 1
        plans += (row_hi - row_lo) * ndiv
        cands += n
        for k in totals:
            totals[k] += counters[k]
    coverage = plans / space.num_plans
    print(f'oracle covered {plans} of {space.num_plans} plans ({100 * coverage:.1f} %), {cands} candidates, '
          f'{done}/{len(items)} work items on {oracle_pool.usable_cores()} cores')
    assert coverage >= 0.25, f'oracle covered only {100 * coverage:.1f} % of the space within {budget} s'
    if done == len(items):
        assert seen.all() and cands == len(rec) == out.summary['num_records']
        assert (totals['B'], totals['runs'], totals['keyerr']) == \
            (out.summary['num_partition_calls'], out.summary['num_balancer_runs'], out.summary['num_keyerror'])


@pytest.mark.parametrize('name', ['c1', 'c2_het16'])
def test_cli_whole_stdout_equals_the_reference_transcript(name, workload_dir, capsys, monkeypatch):
    """The drop-in CLI with METIS_VERBOSE=1 against the stdout captured from the unmodified reference
    (make_golden.py transcript:<name>: print(profile_data), the per-candidate lines of every inter-stage plan,
    len(costs), the ranked table): every line equal, only `search_time:` masked (cost_het_cluster.py:53-80)."""
    _gpu()
    import gzip
    import cost_het_cluster as cli
    from metis_b200.utils import DeviceType
    meta = json.load(open(os.path.join(GOLDEN, f'transcript_{name}.json')))
    gold = gzip.open(os.path.join(GOLDEN, f'transcript_{name}.txt.gz'), 'rt').read().split('\n')
    if name == 'c1':
        argv = ['--model_name', 'GPT', '--model_size', '1.5B', '--num_layers', '10', '--gbs', '128',
                '--max_profiled_tp_degree', '4', '--max_profiled_batch_size', '4', '--min_group_scale_variance', '1',
                '--max_permute_len', '4', '--hidden_size', '4096', '--sequence_length', '1024', '--vocab_size', '51200',
                '--attention_head_size', '32', '--hostfile_path', os.path.join(C1_DIR, 'hostfile'),
                '--clusterfile_path', os.path.join(C1_DIR, 'clusterfile.json'),
                '--profile_data_path', os.path.join(C1_DIR, 'profile_data_samples')]
    else:
        w, root, digest = workload_dir(name)
        assert digest == meta['inputs_sha256']
        argv = w.cli_args(root)
    monkeypatch.setenv('METIS_VERBOSE', '1')
    seqs = [tuple(DeviceType[t] for t in seq) for seq in meta['node_sequences']]
    capsys.readouterr()
    cli.main(argv, node_sequences=seqs, file_order=meta['file_order'])
    ours = capsys.readouterr().out.split('\n')
    ours = ['search_time: <masked>' if ln.startswith('search_time: ') else ln for ln in ours]
    assert len(ours) == len(gold)
    for i, (a, b) in enumerate(zip(ours, gold)):
        assert a == b, f'line {i + 1} differs'


@pytest.mark.parametrize('name,fix', [('mix32', ('Q5',)), ('c2_v100', ('Q6',)), ('mix32', ('Q1', 'Q2', 'Q5', 'Q6'))])
def test_opt_in_corrections_on_gpu_vs_corrected_oracle(name, fix, workload_dir):
    """SURVEY.md 8(f)-4 through the drop-in API: api.cost_het_cluster(..., corrected=fix) equals the oracle run with
    the same corrections (never the default; the strict result is the goldens' business) - every tuple, every cost bit;
    with 'Q5' no partition loses a layer."""
    _gpu()
    from metis_b200 import api
    from oracle import metis_oracle as orc
    meta, arr, call, seqs = _api_inputs(name, workload_dir)
    w, root, _ = workload_dir(name)
    res = api.cost_het_cluster(*call, node_sequences=seqs, device='cuda:0', corrected=fix)
    ocl = orc.OracleCluster(os.path.join(root, 'hostfile'), os.path.join(root, 'clusterfile.json'), corrected=fix)
    oprof, _ = orc.load_profile_dir(os.path.join(root, 'profile'), meta['file_order'])
    omodel = orc.OracleModel(w.num_layers, w.hidden_size, w.sequence_length, w.vocab_size, oprof['model']['parameters'])
    want, counters = orc.het_search(oprof, ocl, omodel, seqs, w.gbs, w.num_layers, w.variance, w.max_permute_len,
                                    w.max_tp, w.max_bs, corrected=fix)
    assert len(res) == len(want) == counters['C']
    assert res.summary['corrected'] == tuple(sorted(fix))
    for g, x in zip(res, want):
        assert g == (x[2], x[3], x[4], x[5], x[6], x[7], x[8])
    if 'Q5' in fix:
        assert all(g[4][-1] == w.num_layers for g in res)


# ---------------------------------------------------------------------------------------------------------------
# SURVEY.md 8(f)-1: device-group rows written by the GPU (het_rows_kernel) = the host enumerator's rows
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('ndev,var,mpl', [(8, 0.5, 4), (16, 1, 6), (32, 0.5, 6), (32, 0, 4), (64, 1, 4), (64, 0.5, 6),
                                          (128, 1, 6), (128, 0, 4), (256, 0, 4)])
def test_rows_written_by_the_gpu_equal_the_host_enumerators(ndev, var, mpl, workload_dir):
    _gpu()
    from metis_b200 import flatten, search
    w, root, _ = workload_dir('sweep_n8_t1')          # any problem: only the candidate space matters here
    cluster, profile, _, cfg = _inputs(root, 'profile', None, w.num_layers, w.hidden_size, w.sequence_length, w.vocab_size)
    seqs = [tuple(w.device_types())]
    problem = flatten.build_problem(profile, cluster, cfg, w.gbs, w.max_tp, w.max_bs, seqs)
    L = 96
    host = flatten.build_plan_space(2, ndev, 64, L, var, mpl)
    dev = flatten.build_plan_space(2, ndev, 64, L, var, mpl, device_rows=True)
    assert dev.comp_recs is not None and dev.rows.size == 0
    assert dev.num_plans == host.num_plans and dev.blocks.tobytes() == host.blocks.tobytes()
    dp = search.DeviceProblem(problem, dev, 'cuda:0')
    assert dp.h2d_bytes == dp._off['rows'][0]                 # the upload stops where the row blob starts
    assert dp.h2d_bytes < 64 * 1024 + 2 * (dev.comp_recs.nbytes + dev.comp_pool.nbytes)
    got = dp.rows_device().cpu().numpy()
    assert got.tobytes() == host.rows[:dev.rows_total_bytes].tobytes()
    # a second upload into the same arena (engine reuse) rewrites the same bytes
    dp.reload(problem, dev)
    dp.upload()
    assert dp.rows_device().cpu().numpy().tobytes() == got.tobytes()


@pytest.mark.parametrize('name', ['mix32', 'c3_homo64_mpl4'])
def test_search_over_gpu_written_rows_gives_the_same_records(name, workload_dir):
    _gpu()
    from metis_b200 import flatten, search
    from metis_b200.workloads import profile_file_order
    w, root, _ = workload_dir(name)
    cluster, profile, _, cfg = _inputs(root, 'profile', profile_file_order(w), w.num_layers, w.hidden_size,
                                       w.sequence_length, w.vocab_size)
    seqs = list(itertools.permutations(w.device_types()))
    problem = flatten.build_problem(profile, cluster, cfg, w.gbs, w.max_tp, w.max_bs, seqs)
    outs = []
    for device_rows in (False, True):
        space = flatten.build_plan_space(len(seqs), cluster.get_total_num_devices(), w.gbs, w.num_layers, w.variance,
                                         w.max_permute_len, device_rows=device_rows)
        dp = search.DeviceProblem(problem, space, 'cuda:0')
        outs.append(search.HetSearcher(dp, want_records=True, want_detail=True).run())
    a, b = outs
    assert len(a.records) > 0 and a.records.tobytes() == b.records.tobytes()
    used = np.arange(a.detail.shape[1])[None, :] < (3 * a.records['num_stage'].astype(np.int64) + 1)[:, None]
    assert (np.where(used, a.detail, 0) == np.where(used, b.detail, 0)).all()     # bytes past 3S+1 are not written


def test_random_small_clusters_on_gpu_vs_oracle(tmp_path):
    """Seeded fuzz through the C ABI: 60 random small clusters (1-3 device types, 2-32 GPUs, odd layer counts and
    batch sizes, tight memories, variance 0 / 0.5 / 1; the generator of the host-build fuzz, another seed), searched
    on the GPU - bulk round forced / chain kernel only, rows from the host enumerator / written by the GPU, in turn -
    and by the oracle: every candidate, counter and fp64 cost bit must agree; a search the oracle aborts with a
    KeyError must report a fatal plan."""
    _gpu()
    from oracle import metis_oracle as orc
    from metis_b200 import flatten, search
    from metis_b200.workloads import materialize, profile_file_order
    from test_device_logic_on_host import _random_workload
    import hostsim_util as hs
    rng = random.Random(20260922)
    done = fatal = candidates = 0
    idx = 0
    while done < 60 and idx < 900:
        idx += 1
        w = _random_workload(rng, idx)
        root = str(tmp_path / w.name)
        materialize(w, root)
        order = profile_file_order(w)
        cluster, profile, _types, cfg = _inputs(root, 'profile', order, w.num_layers, w.hidden_size,
                                                w.sequence_length, w.vocab_size)
        seqs = list(itertools.permutations(w.device_types()))
        ndev = cluster.get_total_num_devices()
        try:
            space = flatten.build_plan_space(len(seqs), ndev, w.gbs, w.num_layers, w.variance, w.max_permute_len,
                                             device_rows=bool(done & 2))
        except IndexError:
            continue
        if not 1 <= space.num_plans <= 6000:
            continue
        problem = flatten.build_problem(profile, cluster, cfg, w.gbs, w.max_tp, w.max_bs, seqs)
        dp = search.DeviceProblem(problem, space, 'cuda:0')
        s = search.HetSearcher(dp, want_records=True, want_detail=True)
        s.shard.reserved = 1 if done & 1 else 2 ** 31 - 1
        out = s.run()
        ocl = orc.OracleCluster(os.path.join(root, 'hostfile'), os.path.join(root, 'clusterfile.json'))
        oprof, _ = orc.load_profile_dir(os.path.join(root, 'profile'), order)
        omodel = orc.OracleModel(w.num_layers, w.hidden_size, w.sequence_length, w.vocab_size, oprof['model']['parameters'])
        try:
            want, counters = orc.het_search(oprof, ocl, omodel, seqs, w.gbs, w.num_layers, w.variance,
                                            w.max_permute_len, w.max_tp, w.max_bs)
        except KeyError:
            assert out.summary['fatal_ordinal'] != 2 ** 64 - 1 and out.summary['fatal_code'] in (1, 2), w
            fatal += 1
            done += 1
            continue
        sm = out.summary
        assert sm['fatal_ordinal'] == 2 ** 64 - 1, w
        assert (space.num_plans, sm['num_partition_calls'], sm['num_balancer_runs'], sm['num_records']) == \
            (counters['A'], counters['B'], counters['runs'], counters['C']), w
        host_space = space if space.rows.size else flatten.build_plan_space(len(seqs), ndev, w.gbs, w.num_layers,
                                                                            w.variance, w.max_permute_len)
        got = hs.unpack_candidates(out.records, out.detail, host_space)
        assert len(got) == len(want), w
        for g, x in zip(got, want):
            assert (g[0], g[1], g[3], g[4], g[5], g[6], g[7]) == (x[0], x[1], x[3], x[4], x[5], x[6], x[7]), (w, g, x)
            assert g[8] == x[8], (w, g[0], g[1], g[8].hex(), x[8].hex())
        candidates += len(want)
        done += 1
    assert done == 60 and candidates > 500, (done, fatal, candidates)
