#!/usr/bin/env python3
"""Generate tests/golden/*.npz by executing the UNMODIFIED reference (/root/reference).

Run in the build container only (the GPU box has no /root/reference):

    PYTHONHASHSEED=0 python tests/golden/make_golden.py [name ...] [--procs 8]

What is reference code and what is harness:
  * every arithmetic / enumeration step is the reference's own classes
    (InterStagePlanGenerator, StagePerformance, IntraStagePlanGenerator,
    LayerLoadBalancer, HeteroCostEstimator, UniformPlanGenerator, HomoCostEstimator);
  * the harness is the loop body of cost_het_cluster.py:25-48 restated so that a
    shard of the inter-stage plans can be evaluated per process, stdout silenced,
    and counters (partition_layer calls, LayerComputeBalancer.run calls) taken by
    wrapping the reference methods;
  * one patch on an in-memory copy: ``utils.DeviceType`` gains H100 and B200
    members (SURVEY.md quirk Q11) - nothing else is changed;
  * the profile file listing order (quirk Q3) is pinned by assigning
    ``loader.profile_data_list`` before ``load_profile_data_all``.

Outputs hold, per costed candidate in ``estimate_costs`` order: inter-stage plan
ordinal, chain step, node-sequence index, device groups, strategies, batches,
layer partition, num_repartition and the fp64 cost (exact bits).
"""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import multiprocessing as mp
import os
import random
import sys
import tempfile
import time
from enum import Enum

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
REF = '/root/reference'
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.dirname(HERE))           # tests/: golden_units, conftest

from metis_b200.workloads import WORKLOADS, Workload, materialize, profile_file_order  # noqa: E402

C1_FLAGS = ['--model_name', 'GPT', '--model_size', '1.5B', '--num_layers', '10', '--gbs', '128',
            '--max_profiled_tp_degree', '4', '--max_profiled_batch_size', '4',
            '--min_group_scale_variance', '1', '--max_permute_len', '4', '--hidden_size', '4096',
            '--sequence_length', '1024', '--vocab_size', '51200', '--attention_head_size', '32']


_REF_CACHE = None


def import_reference():
    """Import the reference with DeviceType extended by H100/B200 (Q11)."""
    global _REF_CACHE
    if _REF_CACHE is not None:
        return _REF_CACHE
    sys.path.insert(0, REF)
    import utils as ref_utils                                   # /root/reference/utils.py

    class DeviceType(Enum):
        A100 = "a100"
        V100 = "v100"
        P100 = "p100"
        T4 = "t4"
        H100 = "h100"
        B200 = "b200"

        @staticmethod
        def from_string(s: str) -> 'DeviceType':
            try:
                return DeviceType[s.upper()]
            except KeyError:
                raise ValueError

    ref_utils.DeviceType = DeviceType
    import arguments, data_loader, gpu_cluster                  # noqa: E401
    from model import cost_estimator, activation_parameter, device_group, load_balancer
    from search_space import plan
    _REF_CACHE = dict(utils=ref_utils, arguments=arguments, data_loader=data_loader, gpu_cluster=gpu_cluster,
                      cost_estimator=cost_estimator, activation_parameter=activation_parameter,
                      device_group=device_group, load_balancer=load_balancer, plan=plan)
    return _REF_CACHE


def build_objects(ref, argv, file_order):
    sys.argv = ['cost_het_cluster.py'] + argv                   # Q7: get_cost re-parses sys.argv
    args = ref['arguments'].parse_args()
    cluster = ref['gpu_cluster'].GPUCluster(hostfile_path=args.hostfile_path,
                                            clusterfile_path=args.clusterfile_path)
    loader = ref['data_loader'].ProfileDataLoader(args.profile_data_path)
    if file_order is not None:
        assert sorted(file_order) == sorted(loader.profile_data_list)
        loader.profile_data_list = list(file_order)
    profile_data, device_types = loader.load_profile_data_all()
    model_config = ref['utils'].ModelConfig(model_name=args.model_name, num_layers=args.num_layers,
                                            sequence_length=args.sequence_length, vocab_size=args.vocab_size,
                                            hidden_size=args.hidden_size,
                                            attention_head_size=args.attention_head_size)
    volume = ref['activation_parameter'].GPTActivationAndParam(model_config, profile_data['model']['parameters'])
    return args, cluster, profile_data, device_types, model_config, volume


def het_shard(job):
    """Evaluate inter-stage plans with ordinal % nshard == shard using reference classes."""
    argv, file_order, node_seq_names, shard, nshard, sample = job
    ref = import_reference()
    args, cluster, profile_data, _, model_config, volume = build_objects(ref, argv, file_order)
    estimator = ref['cost_estimator'].HeteroCostEstimator(profile_data, model_config, volume, cluster)
    balancer = ref['load_balancer'].LayerLoadBalancer(cluster, profile_data, model_config, args.gbs)
    counters = {'A': 0, 'B': 0, 'runs': 0, 'keyerr': 0}
    orig_partition = balancer.partition_layer
    orig_run = ref['load_balancer'].LayerComputeBalancer.run

    def counted_partition(*a, **k):
        counters['B'] += 1
        return orig_partition(*a, **k)

    def counted_run(self):
        counters['runs'] += 1
        return orig_run(self)

    balancer.partition_layer = counted_partition
    ref['load_balancer'].LayerComputeBalancer.run = counted_run
    DeviceType = ref['utils'].DeviceType
    device_set = set(cluster.get_device_types())
    gen = ref['plan'].InterStagePlanGenerator(device_types=device_set,
                                              num_devices=cluster.get_total_num_devices(), gbs=args.gbs,
                                              num_layers=args.num_layers,
                                              variance=args.min_group_scale_variance,
                                              max_permute_len=args.max_permute_len)
    if node_seq_names is not None:      # pin quirk Q4 (set order) to what the parent process saw
        gen.node_sequences = [tuple(DeviceType[n] for n in seq) for seq in node_seq_names]
    rows = []
    fatal = None
    sink = io.StringIO()
    with contextlib.redirect_stdout(sink):
        ordinal = -1
        for inter in gen:
            ordinal += 1
            counters['A'] += 1
            if sample is not None:
                if ordinal not in sample:
                    continue
            elif ordinal % nshard != shard:
                continue
            sink.seek(0)
            sink.truncate(0)
            try:
                perf = ref['device_group'].StagePerformance(model_config, profile_data, cluster, inter)
                rank_map = perf.get_device_placement()
                intra_gen = ref['plan'].IntraStagePlanGenerator(inter, perf, balancer,
                                                                args.max_profiled_tp_degree,
                                                                args.max_profiled_batch_size)
                step = 0
                while intra_gen.has_next:
                    intra = intra_gen.next()
                    try:
                        cost = estimator.get_cost(inter, intra.strategies, intra.layer_partition, rank_map)
                        rows.append((ordinal, step, inter.ns_idx, list(inter.device_groups),
                                     list(intra.strategies), inter.batches, list(intra.layer_partition),
                                     intra.num_repartition, cost, inter.num_stage))
                    except KeyError:
                        counters['keyerr'] += 1
                    step += 1
            except Exception as exc:   # Q8: anything else aborts the reference search
                fatal = (ordinal, type(exc).__name__, str(exc))
                break
    names = [[d.name for d in seq] for seq in gen.node_sequences]
    return rows, counters, fatal, names


def run_het(name, argv, file_order, procs, sample=None):
    t0 = time.time()
    # first a tiny in-process call to learn the node-sequence order this interpreter produces (Q4)
    ref = import_reference()
    args, cluster, *_ = build_objects(ref, argv, file_order)
    gen = ref['plan'].InterStagePlanGenerator(device_types=set(cluster.get_device_types()),
                                              num_devices=cluster.get_total_num_devices(), gbs=args.gbs,
                                              num_layers=args.num_layers,
                                              variance=args.min_group_scale_variance,
                                              max_permute_len=args.max_permute_len)
    node_seq_names = [[d.name for d in seq] for seq in gen.node_sequences]
    sample_set = set(sample) if sample is not None else None
    jobs = [(argv, file_order, node_seq_names, k, procs, sample_set) for k in range(procs)]
    if sample is not None:
        jobs = [(argv, file_order, node_seq_names, 0, 1,
                 set(s for i, s in enumerate(sorted(sample_set)) if i % procs == k)) for k in range(procs)]
    with mp.get_context('fork').Pool(procs) as pool:
        parts = pool.map(het_shard, jobs)
    rows, fatal = [], None
    counters = {'A': parts[0][1]['A'], 'B': 0, 'runs': 0, 'keyerr': 0}
    for r, c, f, _ in parts:
        rows += r
        for k in ('B', 'runs', 'keyerr'):
            counters[k] += c[k]
        if f is not None and (fatal is None or f[0] < fatal[0]):
            fatal = f
    if fatal is not None:
        # the reference stops at the first failing plan: keep only what precedes it
        rows = [r for r in rows if r[0] < fatal[0]]
    rows.sort(key=lambda r: (r[0], r[1]))
    counters['C'] = len(rows)
    wall = time.time() - t0
    print(f'{name}: A={counters["A"]} B={counters["B"]} runs={counters["runs"]} C={counters["C"]} '
          f'keyerr={counters["keyerr"]} fatal={fatal} wall={wall:.1f}s procs={procs}', file=sys.stderr)
    return rows, counters, fatal, node_seq_names, wall


def pack(rows):
    n = len(rows)
    smax = max([len(r[3]) for r in rows], default=1)
    out = {
        'ordinal': np.array([r[0] for r in rows], dtype=np.int64),
        'step': np.array([r[1] for r in rows], dtype=np.int16),
        'ns_idx': np.array([r[2] for r in rows], dtype=np.int16),
        'batches': np.array([r[5] for r in rows], dtype=np.int32),
        'nrep': np.array([r[7] for r in rows], dtype=np.int8),
        'cost': np.array([r[8] for r in rows], dtype=np.float64),
        'label_stage': np.array([r[9] for r in rows], dtype=np.int16),
        'nstage': np.array([len(r[3]) for r in rows], dtype=np.int16),
        'groups': np.zeros((n, smax), dtype=np.uint16),
        'dp': np.zeros((n, smax), dtype=np.uint16),
        'tp': np.zeros((n, smax), dtype=np.uint16),
        'part': np.zeros((n, smax + 1), dtype=np.uint16),
    }
    for i, r in enumerate(rows):
        s = len(r[3])
        out['groups'][i, :s] = r[3]
        out['dp'][i, :s] = [d for d, _ in r[4]]
        out['tp'][i, :s] = [t for _, t in r[4]]
        out['part'][i, :s + 1] = r[6]
    return out


MAX_BYTES = 1_000_000
CANDIDATE_KEYS = ('ordinal', 'step', 'ns_idx', 'batches', 'nrep', 'cost', 'label_stage', 'nstage', 'dp', 'tp', 'part')


def save(name, meta, arrays):
    """Writes tests/golden/<name>.npz without 'groups' (dp * tp; conftest.load_golden rebuilds it).  When the file
    would exceed MAX_BYTES it keeps a seeded sample of the candidates, their positions in 'rows', and records the
    whole list's digest and best in meta (read by conftest.assert_candidates_equal / golden_best)."""
    from conftest import candidates_digest, golden_best
    path = os.path.join(HERE, f'{name}.npz')
    arrays = {k: v for k, v in arrays.items() if k != 'groups'}
    np.savez_compressed(path, meta=np.array(json.dumps(meta)), **arrays)
    n = len(arrays['cost'])
    keep = n
    while os.path.getsize(path) > MAX_BYTES:
        if keep == n:
            meta = dict(meta, best=list(golden_best({}, arrays)),
                        digest=candidates_digest(arrays['ordinal'], arrays['step'], arrays['nrep'], arrays['nstage'],
                                                 arrays['cost'], arrays['dp'], arrays['tp'], arrays['part']))
        keep = int(keep * 0.95 * MAX_BYTES / os.path.getsize(path))
        rows = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        sub = {k: (v[rows] if k in CANDIDATE_KEYS else v) for k, v in arrays.items()}
        np.savez_compressed(path, meta=np.array(json.dumps(meta)), rows=rows, **sub)
    print(f'wrote {path} ({os.path.getsize(path)} bytes, {keep} of {n} candidates)', file=sys.stderr)


def stratified_sample(w: Workload, fraction: float, seed: int = 4321):
    """Ordinals covering EVERY (node sequence, stage count) block of the plan space - its first two and its last
    device-group rows with every divisor of gbs, which includes every mislabelled Q1 block - plus a uniform
    `fraction` of all ordinals.  The block structure comes from the library's host enumerator (it only defines
    WHICH plans the reference is asked to evaluate; what the reference returns for them is its own)."""
    import math
    from metis_b200 import flatten
    nseq = math.factorial(len(w.device_types()))
    ndev = sum(n for _, n in w.nodes)
    space = flatten.build_plan_space(nseq, ndev, w.gbs, w.num_layers, w.variance, w.max_permute_len)
    ndiv = len(space.batches)
    picks = set()
    for blk in space.blocks:
        first, rows = int(blk['first_ordinal']), int(blk['num_rows'])
        for row in sorted({0, 1, rows // 2, rows - 1}):
            if 0 <= row < rows:
                picks.update(range(first + row * ndiv, first + (row + 1) * ndiv))
    rng = random.Random(seed)
    total = space.num_plans
    picks.update(rng.sample(range(total), int(total * fraction)))
    return sorted(picks), total


def golden_het_workload(w: Workload, procs: int, sample_n: int = 0, strat: float = 0.0):
    with tempfile.TemporaryDirectory() as root:
        digest = materialize(w, root)
        order = profile_file_order(w)
        argv = w.cli_args(root)
        sample = None
        if strat:
            sample, _total = stratified_sample(w, strat)
        if sample_n:
            # count plans with the reference generator, then sample ordinals with a fixed seed
            ref = import_reference()
            args, cluster, *_ = build_objects(ref, argv, order)
            gen = ref['plan'].InterStagePlanGenerator(device_types=set(cluster.get_device_types()),
                                                      num_devices=cluster.get_total_num_devices(),
                                                      gbs=args.gbs, num_layers=args.num_layers,
                                                      variance=args.min_group_scale_variance,
                                                      max_permute_len=args.max_permute_len)
            total = sum(1 for _ in gen)
            picks = set(random.Random(1234).sample(range(total), min(sample_n, total)))
            nseq = len(gen.node_sequences)
            for k in range(1, nseq):       # plus a window at the start of every later node sequence:
                start = k * (total // nseq) - 64      # mislabelled Q1 blocks and mixed-type stages
                picks.update(range(max(0, start), min(total, start + 1200)))
            sample = sorted(picks)
        rows, counters, fatal, names, wall = run_het(w.name, argv, order, procs, sample)
        meta = {'workload': w.name, 'inputs_sha256': digest, 'file_order': order, 'node_sequences': names,
                'counters': counters, 'fatal': fatal, 'reference_wall_s': wall, 'procs': procs,
                'sampled_ordinals': sample is not None, 'python': sys.version.split()[0]}
        arrays = pack(rows)
        if sample is not None:
            arrays['sample'] = np.array(sample, dtype=np.int64)
        save(w.name, meta, arrays)


def golden_c1(procs: int):
    """BASELINE configs[0]: shipped hostfile/clusterfile/profile_data_samples, het + homo paths."""
    fix = os.path.join(HERE, 'fixtures', 'c1')
    order = sorted(os.listdir(os.path.join(REF, 'profile_data_samples')))
    # use the listing order the survey measured (first file tp2_bs2) to reproduce KAT-1 digits
    order = ['DeviceType.A100_tp2_bs2.json'] + [f for f in order if f != 'DeviceType.A100_tp2_bs2.json']
    argv = C1_FLAGS + ['--hostfile_path', os.path.join(fix, 'hostfile'),
                       '--clusterfile_path', os.path.join(fix, 'clusterfile.json'),
                       '--profile_data_path', os.path.join(fix, 'profile_data_samples')]
    rows, counters, fatal, names, wall = run_het('c1_het', argv, order, 1)
    meta = {'workload': 'c1_het', 'file_order': order, 'node_sequences': names, 'counters': counters,
            'fatal': fatal, 'reference_wall_s': wall, 'procs': 1, 'flags': C1_FLAGS}
    save('c1_het', meta, pack(rows))

    # homo path: harness around the untouched cost_homo_cluster() (its __main__ is broken as shipped)
    ref = import_reference()
    sys.path.insert(0, REF)
    import cost_homo_cluster as homo_mod
    args, cluster, profile_data, device_types, model_config, volume = build_objects(ref, argv, order)
    estimator = ref['cost_estimator'].HomoCostEstimator(profile_data, model_config, volume, cluster)
    homo_mod.device_types = device_types
    yielded = sum(1 for _ in ref['plan'].UniformPlanGenerator(cluster.get_total_num_devices(),
                                                              args.max_profiled_tp_degree, args.gbs))
    with contextlib.redirect_stdout(io.StringIO()):
        costs = homo_mod.cost_homo_cluster(args, cluster, estimator)
    arr = {'plan': np.array([[p.dp, p.pp, p.tp, p.mbs, p.gbs] for p, _ in costs], dtype=np.int32),
           'cost': np.array([c for _, c in costs], dtype=np.float64)}
    meta = {'workload': 'c1_homo', 'file_order': order, 'yielded': yielded, 'costed': len(costs), 'flags': C1_FLAGS}
    save('c1_homo', meta, arr)
    print(f'c1_homo: yielded={yielded} costed={len(costs)} best={min(c for _, c in costs)!r}', file=sys.stderr)


def golden_homo_workload(w: Workload):
    """cost_homo_cluster() of the reference on a synthetic single-type workload."""
    with tempfile.TemporaryDirectory() as root:
        digest = materialize(w, root)
        order = profile_file_order(w)
        argv = w.cli_args(root)
        ref = import_reference()
        sys.path.insert(0, REF)
        import cost_homo_cluster as homo_mod
        args, cluster, profile_data, device_types, model_config, volume = build_objects(ref, argv, order)
        estimator = ref['cost_estimator'].HomoCostEstimator(profile_data, model_config, volume, cluster)
        homo_mod.device_types = device_types
        yielded = sum(1 for _ in ref['plan'].UniformPlanGenerator(cluster.get_total_num_devices(),
                                                                  args.max_profiled_tp_degree, args.gbs))
        with contextlib.redirect_stdout(io.StringIO()):
            costs = homo_mod.cost_homo_cluster(args, cluster, estimator)
        arr = {'plan': np.array([[p.dp, p.pp, p.tp, p.mbs, p.gbs] for p, _ in costs], dtype=np.int32).reshape(-1, 5),
               'cost': np.array([c for _, c in costs], dtype=np.float64)}
        meta = {'workload': w.name, 'inputs_sha256': digest, 'file_order': order, 'yielded': yielded,
                'costed': len(costs)}
        save(w.name + '_homo', meta, arr)
        print(f'{w.name}_homo: yielded={yielded} costed={len(costs)}', file=sys.stderr)


def golden_transcript(name: str):
    """The reference's WHOLE stdout for one configuration (cost_het_cluster.py:53-80, with the per-candidate lines of
    plan.py / load_balancer.py / cost_estimator.py): the unmodified cost_het_cluster() function driven exactly like the
    reference's __main__ block, with the profile listing order pinned (Q3) and PYTHONHASHSEED=0 (Q4).  The
    `search_time:` line is masked.  -> tests/golden/transcript_<name>.txt.gz + .json (flags, node sequences)"""
    import gzip
    ref = import_reference()
    sys.path.insert(0, REF)
    import cost_het_cluster as ref_main                         # /root/reference/cost_het_cluster.py
    with tempfile.TemporaryDirectory() as root:
        if name == 'c1':
            fix = os.path.join(HERE, 'fixtures', 'c1')
            order = sorted(os.listdir(os.path.join(fix, 'profile_data_samples')))
            order = ['DeviceType.A100_tp2_bs2.json'] + [f for f in order if f != 'DeviceType.A100_tp2_bs2.json']
            argv = C1_FLAGS + ['--hostfile_path', os.path.join(fix, 'hostfile'),
                               '--clusterfile_path', os.path.join(fix, 'clusterfile.json'),
                               '--profile_data_path', os.path.join(fix, 'profile_data_samples')]
            digest = None
        else:
            w = WORKLOADS[name]
            digest = materialize(w, root)
            order = profile_file_order(w)
            argv = w.cli_args(root)
        args, cluster, profile_data, _types, model_config, volume = build_objects(ref, argv, order)
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            print(profile_data)
            estimator = ref['cost_estimator'].HeteroCostEstimator(profile_data, model_config, volume, cluster)
            balancer = ref['load_balancer'].LayerLoadBalancer(cluster, profile_data, model_config, args.gbs)
            t0 = time.time()
            costs = ref_main.cost_het_cluster(args, cluster, profile_data, model_config, estimator, balancer)
            print(f'search_time: {time.time() - t0}s')
            print(f'len(costs): {len(costs)}')
            ranked = sorted(costs, key=lambda kv: kv[6])
            print('rank, cost, node_sequence, device_groups, strategies(dp_deg, tp_deg), batches(number of batch), layer_partition')
            for idx, result in enumerate(ranked):
                print(f'{idx + 1}, {result[6]}, {result[0]}, {result[1]}, {result[2]}, {result[3]}, {result[4]}')
        text = buf.getvalue()
        text = '\n'.join('search_time: <masked>' if ln.startswith('search_time: ') else ln for ln in text.split('\n'))
        gen = ref['plan'].InterStagePlanGenerator(device_types=set(cluster.get_device_types()),
                                                  num_devices=cluster.get_total_num_devices(), gbs=args.gbs,
                                                  num_layers=args.num_layers, variance=args.min_group_scale_variance,
                                                  max_permute_len=args.max_permute_len)
        names = [[d.name for d in seq] for seq in gen.node_sequences]
    with gzip.open(os.path.join(HERE, f'transcript_{name}.txt.gz'), 'wt') as fh:
        fh.write(text)
    json.dump({'workload': name, 'inputs_sha256': digest, 'file_order': order, 'node_sequences': names,
               'costs': len(costs), 'lines': text.count('\n')},
              open(os.path.join(HERE, f'transcript_{name}.json'), 'w'))
    print(f'transcript_{name}: {len(costs)} costs, {text.count(chr(10))} lines, {len(text)} bytes', file=sys.stderr)


def golden_units():
    """Unit-level vectors from reference functions on seeded random inputs."""
    ref = import_reference()
    from search_space.device_group import gen_dgroups_for_stages_with_variance, gen_device_group_shapes
    # device-group rows: full tables for small cases
    dg = []
    for ndev in (4, 8, 16, 32):
        for variance in (0, 1):
            for mpl in (2, 4, 6):
                for stages in range(1, min(ndev, 12) + 1):
                    rows = gen_dgroups_for_stages_with_variance(stages, ndev, gen_device_group_shapes(ndev),
                                                                variance, mpl)
                    dg.append({'ndev': ndev, 'variance': variance, 'mpl': mpl, 'stages': stages, 'rows': rows})
    # LayerComputeBalancer.run and _adj_compute_performance on the seeded inputs of tests/golden_units.py; only the
    # outputs are stored
    from golden_units import unit_inputs
    bal_in, adj_in = unit_inputs()
    LCB = ref['load_balancer'].LayerComputeBalancer
    bal = [LCB(S, L, list(capa), lc).run()[0] for S, L, capa, lc in bal_in]
    llb_cls = ref['load_balancer'].LayerLoadBalancer
    dummy = llb_cls.__new__(llb_cls)
    adj = []
    with contextlib.redirect_stdout(io.StringIO()):
        for c, mc, md in adj_in:
            out = dummy._adj_compute_performance(list(c), list(mc), list(md))
            adj.append(None if out is None else [x.hex() for x in out])
    path = os.path.join(HERE, 'units.json')
    import gzip
    with gzip.GzipFile(path + '.gz', 'wb', mtime=0) as fh:
        fh.write(json.dumps({'device_groups': dg, 'balancer_part': bal, 'adjust_out': adj}).encode())
    print(f'wrote {path}.gz', file=sys.stderr)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('names', nargs='*')
    ap.add_argument('--procs', type=int, default=8)
    ns = ap.parse_args()
    sys.argv = sys.argv[:1]
    if os.environ.get('PYTHONHASHSEED') != '0':
        os.environ['PYTHONHASHSEED'] = '0'
        os.execv(sys.executable, [sys.executable] + [os.path.abspath(__file__)] + ns.names + ['--procs', str(ns.procs)])
    todo = ns.names or ['units', 'c1', 'c2_het16', 'c2_v100', 'mix32', 'het32_tight', 'fatal_gbs96']
    for name in todo:
        if name == 'units':
            golden_units()
        elif name == 'c1':
            golden_c1(ns.procs)
        elif name.startswith('transcript:'):
            golden_transcript(name.split(':', 1)[1])
        elif name.endswith(':homo'):
            golden_homo_workload(WORKLOADS[name.split(':')[0]])
        elif name.endswith(':sample'):
            golden_het_workload(WORKLOADS[name.split(':')[0]], ns.procs, sample_n=20000)
        elif ':strat' in name:            # name:strat=0.05 -> every block + 5 % of the ordinals
            base, _, frac = name.partition(':strat')
            golden_het_workload(WORKLOADS[base], ns.procs, strat=float(frac.lstrip('=') or 0.01))
        else:
            golden_het_workload(WORKLOADS[name], ns.procs)


if __name__ == '__main__':
    main()
