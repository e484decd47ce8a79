#!/usr/bin/env python3
"""bench.py - candidate plans evaluated / second on B200 (BASELINE.json metric).

A "step" is one full search of the workload's candidate space (every inter-stage plan enumerated by
InterStagePlanGenerator, its intra-stage chain, load balancer and cost model) by libmetis_b200.so.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl reference] [--dump-outputs DIR]

Workload: BASELINE.json configs[2] ("homo 64-GPU cluster, 96-layer GPT-3, gbs=512 (~10^6 candidates)
- 1xB200, HBM-roofline capture"), i.e. c3_homo64_mpl6 = 771 750 inter-stage plans, the configuration the
metric is quoted on for one GPU; configs[1] (16 GPUs, 1 752 plans) is a parity-test case
(tests/test_gpu_parity.py).  N > 1 shards the same space by plan ordinal over the ranks (strong scaling)
with one NCCL all_gather of 32-byte best records per step.

Timed regions
  value : tables + plan space already resident in HBM; per step CUDA events on the launching stream around
          pack + admission + sort + bulk round + chain kernel + finalize, every costed candidate's 16-byte
          record written to HBM (+ the NCCL exchange when N > 1); a 256 MiB write between steps flushes L2;
          ms_per_step = mean, max over ranks.
  e2e   : per step one call of the drop-in function the reference's callers use,
          metis_b200.api.cost_het_cluster(args, gpu_cluster, profile_data, model_config, cost_estimator,
          layer_load_balancer) - exactly the call cost_het_cluster.py:71-74 times - from HOST inputs (nested
          profile dicts, cluster object): flattening, host enumeration of the plan space (C++), one H2D copy
          of every table from pinned memory, the kernels, device sort, D2H of all 16-byte records and of the
          ranking permutation, then len(result) and result.best() (strategies + partition of the winner);
          wall clock between device synchronisations, max over ranks.
  cpu_baseline / --impl reference : the reference's CPU implementation of the path on a bounded uniform sample
          of the same plans, one process per usable host core: the unmodified reference from baseline/_ref when
          that directory exists (kind "reference"), else the oracle (Python port of the pure-Python reference,
          oracle/metis_oracle.py, kind "port").

--steps K sets the number of timed steps of every timed region: `value` and `e2e` of the headline workload and of
each workload under `extra` (so a default run makes K end-to-end calls of the 68 M-plan configs[3] space too).

--dump-outputs DIR writes, after the timed steps, what the last `value` search of the headline workload computed
(the workloads under `extra` are not written): the costed candidates' records (records_cost, records_ordinal,
records_step, records_num_repartition, records_num_stage, sorted by ordinal and step), counters and best, as float64
.npy files.  The workloads are seeded, so two builds run with the same arguments can be compared file for file.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

import numpy as np  # noqa: E402

METRIC = 'candidate plans evaluated/sec'
DEFAULT_WORKLOAD = 'c3_homo64_mpl6'
EXTRA_WORKLOADS = ('c4_het128', 'c4_het128_mpl6')       # BASELINE configs[3] at max_permute_len 4 and 6
REF_DIR = os.path.join(REPO, 'baseline', '_ref')
DUMP_BYTES = 64_000_000                                   # --dump-outputs: at most this much in all


def usable_cores():
    """(threads this process may run on, cgroup CPU quota in cores or None)."""
    try:
        aff = len(os.sched_getaffinity(0))
    except AttributeError:
        aff = os.cpu_count() or 1
    quota = None
    try:
        txt = open('/sys/fs/cgroup/cpu.max').read().split()
        if txt[0] != 'max':
            quota = float(txt[0]) / float(txt[1])
    except Exception:
        try:
            q = int(open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us').read())
            p = int(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
            if q > 0:
                quota = q / p
        except Exception:
            pass
    return aff, quota


# ---------------------------------------------------------------------------------------------
# CPU side: the reference's implementation on a bounded sample (cpu_baseline and --impl reference)
# ---------------------------------------------------------------------------------------------
_W = {}


def _cpu_worker_init(workload_name, root, share_seed, nproc, per_step, nsteps, use_ref):
    """Each worker loads the inputs and collects ITS sampled plans (untimed)."""
    import itertools
    from metis_b200.workloads import WORKLOADS, profile_file_order
    w = WORKLOADS[workload_name]
    _W.update(w=w, per_step=per_step, share=(share_seed, nproc, nsteps), use_ref=use_ref, root=root)
    if use_ref:
        return
    from oracle import metis_oracle as orc
    cluster = orc.OracleCluster(os.path.join(root, 'hostfile'), os.path.join(root, 'clusterfile.json'))
    profile, _ = orc.load_profile_dir(os.path.join(root, 'profile'), profile_file_order(w))
    model = orc.OracleModel(w.num_layers, w.hidden_size, w.sequence_length, w.vocab_size,
                            profile['model']['parameters'])
    seqs = list(itertools.permutations(w.device_types()))
    _W.update(orc=orc, cluster=cluster, profile=profile, model=model, norm=orc.norm_layer_duration(profile),
              plans={}, seqs=seqs)


def _my_sample(worker, total):
    import random
    seed, nproc, nsteps = _W['share']
    want = random.Random(seed).sample(range(total), min(total, nproc * nsteps * _W['per_step']))
    return {o: (i // nproc) % nsteps for i, o in enumerate(want) if i % nproc == worker}   # ordinal -> step index


def _cpu_worker_collect(args):
    worker, total = args
    mine = _my_sample(worker, total)
    if _W['use_ref']:
        _W['mine'] = mine
        return len(mine)
    orc, w = _W['orc'], _W['w']
    plans = {}
    for ordinal, plan in enumerate(orc.inter_stage_plans(_W['seqs'], _W['cluster'].total_devices, w.gbs,
                                                         w.num_layers, w.variance, w.max_permute_len)):
        if ordinal in mine:
            plans.setdefault(mine[ordinal], []).append((ordinal, dict(plan, device_groups=list(plan['device_groups']))))
    _W['plans'] = plans
    return sum(len(v) for v in plans.values())


def _cpu_worker_step(step):
    w = _W['w']
    if _W['use_ref']:
        return _ref_worker_step(step)
    orc = _W['orc']
    counters = {'A': 0, 'B': 0, 'C': 0, 'runs': 0, 'keyerr': 0}
    out = []
    t0 = time.perf_counter()
    for ordinal, plan in _W['plans'].get(step, []):
        counters['A'] += 1
        orc.het_evaluate_plan(_W['profile'], _W['cluster'], _W['model'], _W['norm'], plan, ordinal, w.num_layers,
                              w.max_tp, w.max_bs, counters, out)
    return counters['A'], counters['C'], time.perf_counter() - t0


def _ref_worker_step(step):
    """The unmodified reference (baseline/_ref) on this worker's sampled ordinals of `step`, driven like
    cost_het_cluster.py:25-48 (tests/golden/make_golden.py het_shard; enumeration of the skipped plans is inside
    the timed region, like in the reference's own loop)."""
    from tests.golden import make_golden as mg
    from metis_b200.workloads import profile_file_order
    mg.REF = REF_DIR
    w = _W['w']
    sample = {o for o, s in _W['mine'].items() if s == step}
    t0 = time.perf_counter()
    rows, counters, _fatal, _names = mg.het_shard((w.cli_args(_W['root']), profile_file_order(w), None, 0, 1, sample))
    return len(sample), len(rows), time.perf_counter() - t0


class CpuArm:
    """Pool of reference workers over a bounded sample of the workload's plans."""

    def __init__(self, workload_name, total_plans, per_step_per_core, nsteps):
        import multiprocessing as mp
        from metis_b200.workloads import WORKLOADS, materialize
        aff, quota = usable_cores()
        self.affinity, self.quota = aff, quota
        self.cores = max(1, min(aff, int(quota)) if quota else aff)
        self.kind = 'reference' if os.path.exists(os.path.join(REF_DIR, 'cost_het_cluster.py')) else 'port'
        self.tmp = tempfile.TemporaryDirectory()
        materialize(WORKLOADS[workload_name], self.tmp.name)
        self.pool = mp.get_context('spawn').Pool(self.cores, initializer=_cpu_worker_init,
                                                 initargs=(workload_name, self.tmp.name, 20240921, self.cores,
                                                           per_step_per_core, nsteps, self.kind == 'reference'))
        self.collected = sum(self.pool.map(_cpu_worker_collect, [(k, total_plans) for k in range(self.cores)], 1))
        self.per_process = []

    def step(self, idx):
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_worker_step, [idx] * self.cores, 1)
        wall = time.perf_counter() - t0
        self.per_process += [r[0] / r[2] for r in res if r[2] > 0]
        return sum(r[0] for r in res), sum(r[1] for r in res), wall

    def describe(self, plans, costed, total, wall):
        impl = 'unmodified reference (baseline/_ref)' if self.kind == 'reference' else \
            'oracle/metis_oracle.py (Python port of the pure-Python reference)'
        pp = sorted(self.per_process)
        return (f'{plans} uniformly sampled inter-stage plans of the same {total}-plan space ({costed} costed), {impl}, '
                f'{self.cores} processes (sched_getaffinity {self.affinity}, cgroup quota {self.quota}), {wall:.1f} s; '
                f'plans/s per process min/median/max {pp[0]:.0f}/{pp[len(pp) // 2]:.0f}/{pp[-1]:.0f}' if pp else '')

    def close(self):
        self.pool.close()
        self.pool.join()
        self.tmp.cleanup()


def count_plans_oracle(workload_name):
    """A (number of inter-stage plans) with the oracle's generator - no library, no GPU (reference arm)."""
    import itertools
    from metis_b200.workloads import WORKLOADS
    from oracle import metis_oracle as orc
    w = WORKLOADS[workload_name]
    seqs = list(itertools.permutations(w.device_types()))
    ndev = sum(n for _, n in w.nodes)
    return sum(1 for _ in orc.inter_stage_plans(seqs, ndev, w.gbs, w.num_layers, w.variance, w.max_permute_len))


def run_reference_arm(ns):
    """--impl reference: the reference's CPU implementation of the path, all usable host cores, rank 0 only."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    total = count_plans_oracle(ns.workload)
    steps, warm = ns.steps, ns.warmup
    budget_s = 150.0
    per_step = max(40, int(budget_s / (steps + warm) * 350))           # ~350 plans/s/core in CPython
    arm = CpuArm(ns.workload, total, per_step, steps + warm)
    for i in range(warm):
        arm.step(i)
    arm.per_process = []
    plans = costed = 0
    wall = 0.0
    for i in range(warm, warm + steps):
        a, c, t = arm.step(i)
        plans, costed, wall = plans + a, costed + c, wall + t
    sample = arm.describe(plans, costed, total, wall)
    arm.close()
    value = plans / wall
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': 'plans/s', 'n_gpus': ns.gpus,
        'steps': steps, 'warmup': warm, 'ms_per_step': 1e3 * wall / steps, 'higher_is_better': True,
        'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': workload_config(ns.workload, total),
        'cpu_baseline': {'value': value, 'unit': 'plans/s', 'cores': arm.cores, 'kind': arm.kind, 'sample': sample},
        'e2e': {'value': value, 'unit': 'plans/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'costed_per_s': costed / wall,
    }
    emit_result(line)


def workload_config(name, num_plans):
    from metis_b200.workloads import WORKLOADS
    w = WORKLOADS[name]
    return {'workload': f'{name}: {len(w.nodes)} nodes x {w.nodes[0][1]} GPUs ({"+".join(w.device_types())}), '
                        f'{w.num_layers} layers, gbs {w.gbs}, variance {w.variance}, max_permute_len '
                        f'{w.max_permute_len}, tp<= {w.max_tp}, bs<= {w.max_bs} (BASELINE.json configs[2])',
            'inter_stage_plans': int(num_plans), 'l2': 'flushed between timed steps (256 MiB write)',
            'parallelism': 'plans sharded by ordinal, interleaved 128-plan tiles'}


# ---------------------------------------------------------------------------------------------
# GPU side
# ---------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Streams `nvidia-smi -lms 50` for one GPU while the timed regions run (B200_PROFILING.md clocks line)."""

    QUERY = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.proc = None
        self.armed = threading.Event()

    def run(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.index}', f'--query-gpu={self.QUERY}',
                                          '--format=csv,noheader,nounits', '-lms', '50'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.armed.is_set() and line.strip():
                    self.rows.append([x.strip() for x in line.strip().split(',')])
        except Exception:
            pass

    def stop(self):
        self.armed.clear()
        if self.proc is not None:
            self.proc.terminate()

    def summary(self):
        if not self.rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        sm = [float(r[0]) for r in self.rows if r[0].replace('.', '').isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith('active') for r in self.rows)]
        return {'sm_mhz': statistics.median(sm) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': reasons, 'samples': len(self.rows),
                'window': 'device-timed steps + end-to-end steps (both keep the GPU busy)'}


def dump_outputs(out_dir, searcher):
    """What the searcher's last search computed, as HetSearcher.run hands it to a caller: every costed candidate's
    record in estimate_costs order (ordinal, then chain step), the counters and the best record, each as float64
    (exact for these integers).  More than DUMP_BYTES of records are cut to a seeded sample of positions in that
    order, whose indices are written too."""
    from metis_b200 import native
    sm = searcher.summary()
    n = int(sm.num_records)
    rec = searcher.records[:2 * n].cpu().numpy().view(native.RECORD_DTYPE)
    rec = rec[np.lexsort((rec['step'], rec['ordinal']))]
    fields = ('cost', 'ordinal', 'step', 'num_repartition', 'num_stage')
    keep = (DUMP_BYTES - 4096) // (8 * (len(fields) + 1))    # 4 KiB for the small arrays and the .npy headers
    out = {}
    if n > keep:
        idx = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        rec = rec[idx]
        out['records_index'] = idx.astype(np.float64)
    for f in fields:
        out[f'records_{f}'] = rec[f].astype(np.float64)
    out['counters'] = np.array([sm.num_records, sm.num_partition_calls, sm.num_balancer_runs, sm.num_keyerror],
                               dtype=np.float64)
    b = sm.best
    out['best'] = np.array([b.cost, b.ordinal, b.step, b.num_repartition, b.num_stage] if n else [np.nan] * 5,
                           dtype=np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in out.items():
        np.save(os.path.join(out_dir, f'{name}.npy'), arr)


def run_ours(ns, emit=True, dump_dir=None):
    """One workload; rank 0 returns the JSON line (and prints it when ``emit``); with ``dump_dir`` every rank writes
    the outputs of its last timed search there."""
    import torch
    import torch.distributed as dist
    from metis_b200 import api, flatten, native, search
    from metis_b200.arguments import parse_args
    from metis_b200.data_loader import ProfileDataLoader
    from metis_b200.gpu_cluster import GPUCluster
    from metis_b200.utils import ModelConfig
    from metis_b200.workloads import WORKLOADS, materialize, profile_file_order
    import itertools

    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm')
    native.load_library()
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device(f'cuda:{local}')
    if world > 1 and not dist.is_initialized():
        dist.init_process_group('nccl', device_id=dev)
    assert world == ns.gpus or world == 1 and ns.gpus == 1, f'--gpus {ns.gpus} but WORLD_SIZE {world}'

    # ---- host inputs, built exactly like cost_het_cluster.py:53-69 builds them ---------------------
    w = WORKLOADS[ns.workload]
    tmp = tempfile.TemporaryDirectory()
    materialize(w, tmp.name)
    args = parse_args(w.cli_args(tmp.name))
    cluster = GPUCluster(args.hostfile_path, args.clusterfile_path)
    profile, _ = ProfileDataLoader(args.profile_data_path, profile_file_order(w)).load_profile_data_all()
    cfg = ModelConfig(model_name=args.model_name, num_layers=args.num_layers, sequence_length=args.sequence_length,
                      vocab_size=args.vocab_size, hidden_size=args.hidden_size, attention_head_size=args.attention_head_size)
    volume = api.GPTActivationAndParam(cfg, profile['model']['parameters'])
    estimator = api.HeteroCostEstimator(profile, cfg, volume, cluster)
    balancer = api.LayerLoadBalancer(cluster, profile, cfg, args.gbs)
    seqs = list(itertools.permutations(w.device_types()))

    def api_call():
        return api.cost_het_cluster(args, cluster, profile, cfg, estimator, balancer, node_sequences=seqs, device=dev)

    # ---- device-resident problem for `value` -----------------------------------------------------
    t0 = time.perf_counter()
    problem, space, _ = api.het_problem(args, cluster, profile, cfg, balancer, seqs, device_rows=True)
    host_prep_s = time.perf_counter() - t0
    dp = search.DeviceProblem(problem, space, dev)
    tile = 128
    probe = search.HetSearcher(dp, rank, world, tile, want_records=True, want_detail=False)
    stream = torch.cuda.current_stream(dev)
    ref = probe.run(stream)                                   # sizes the record buffer, proves the result
    if ref.summary['fatal_ordinal'] != 2 ** 64 - 1:
        raise SystemExit(f'fatal plan {ref.summary}')
    full = search.HetSearcher(dp, rank, world, tile, want_records=True, want_detail=False,
                              capacity=len(ref.records) + 1024)     # `value`: every record written to HBM
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def exchange(best):
        return search.global_best(best, dev) if world > 1 else best

    def gpu_step():
        full.launch(stream)
        if world > 1:
            # the summary lands in pinned memory after the stream sync; the collective itself is tiny
            stream.synchronize()
            sm = full.summary()
            b = sm.best
            lb = (b.cost, b.ordinal, b.step, b.num_repartition, b.num_stage) if sm.num_records else None
            return exchange(lb)
        return None

    for _ in range(max(ns.warmup, 3)):
        gpu_step()
    stream.synchronize()
    if world > 1:
        counters = search.global_counters(ref.summary, dev)
        gbest = exchange(ref.best)
    else:
        counters, gbest = ref.summary, ref.best

    # ---- timed: K steps, device events, L2 flushed between steps ---------------------------------
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()                  # nvidia-smi is already streaming when the timed region starts
        time.sleep(0.3)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    if sampler:
        sampler.armed.set()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(ns.steps)]
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(ns.steps)]
    for a, b in kev:
        a.record(stream)
        b.record(stream)           # creates the handles; the library re-records them around the search kernels
    wall0 = time.perf_counter()
    for i in range(ns.steps):
        flush.fill_(i & 0xFF)
        ev[i][0].record(stream)
        dp.lib.metis_set_profile_events(kev[i][0].cuda_event, kev[i][1].cuda_event)
        gpu_step()
        ev[i][1].record(stream)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    wall = time.perf_counter() - wall0
    step_ms = [a.elapsed_time(b) for a, b in ev]
    kern_ms = [a.elapsed_time(b) for a, b in kev]
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    kmean = torch.tensor([sum(kern_ms) / len(kern_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(kmean, op=dist.ReduceOp.MAX)
    ms_per_step = float(total_ms.item()) / ns.steps
    kernel_ms = float(kmean.item())
    if dump_dir:
        dump_outputs(dump_dir if world == 1 else os.path.join(dump_dir, f'rank{rank}'), full)

    # ---- e2e: the drop-in API call from host inputs, every step -----------------------------------
    e2e_steps = ns.steps
    e2e_wall, parts = [], []
    res = None
    for i in range(e2e_steps + 2):                            # two warm-up calls: engine creation, buffer growth
        flush.fill_(i)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        res = api_call()
        n_res = len(res)
        best = res.best()
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        if i >= 2:
            e2e_wall.append(dt)
            parts.append(res.timings)
        assert n_res == counters['num_records'] and best is not None and best[6] == gbest[0], (n_res, best, gbest)
    e2e_t = torch.tensor([statistics.mean(e2e_wall)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_s = float(e2e_t.item())
    if sampler:
        sampler.armed.clear()
        sampler.stop()
        sampler.join(timeout=3)

    A = space.num_plans
    if rank == 0:
        nst = space.blocks['num_stage'].astype(np.int64)
        plans_per_block = space.blocks['num_rows'].astype(np.int64) * len(space.batches)
        alg_bytes = int((plans_per_block * (nst + 16)).sum() + 16 * counters['num_records'])
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(REPO, 'MEASURED_PEAKS.json')))
        except Exception:
            pass
        peak = float(peaks.get('hbm_gbs', 6650.0))
        achieved = alg_bytes / world / (kernel_ms * 1e-3) / 1e9
        traffic = None                                        # measured for the 1-GPU launch only
        tpath = os.path.join(REPO, 'profiles', 'r02_traffic.json')
        if os.path.exists(tpath) and world == 1:
            traffic = json.load(open(tpath)).get('dram_bytes_per_search')
        eng = api._ENGINES.get((local, rank, world))
        h2d = int(eng[0].h2d_bytes) if eng else int(dp.h2d_bytes)
        n_rec = counters['num_records'] if world > 1 else len(ref.records)
        # all records + summary + the winner's detail row and device-group row (the ranking permutation is computed and
        # copied only when ranked() is asked for - the reference's caller sorts, not the function)
        d2h = 16 * n_rec + 96 + (3 * int(nst.max()) + 1) + int(nst.max())
        mean_part = {k: 1e3 * statistics.mean(p[k] for p in parts) for k in parts[0]} if parts else {}
        line = {
            'metric': METRIC, 'value': A / (ms_per_step * 1e-3), 'unit': 'plans/s', 'n_gpus': world,
            'steps': ns.steps, 'warmup': max(ns.warmup, 3), 'ms_per_step': ms_per_step, 'higher_is_better': True,
            'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': workload_config(ns.workload, A),
            'counters': {'A_inter_stage_plans': A, 'B_partition_layer_calls': counters['num_partition_calls'],
                         'balancer_runs': counters['num_balancer_runs'], 'C_costed': counters['num_records'],
                         'keyerror': counters['num_keyerror'], 'admitted_rank0': ref.summary['num_admitted'],
                         'chained_rank0': ref.summary['num_chained']},
            'best_plan': {'cost': gbest[0], 'ordinal': gbest[1], 'step': gbest[2]} if gbest else None,
            'costed_per_s': counters['num_records'] / (ms_per_step * 1e-3),
            'time_to_best_ms': {'gpu_resident': ms_per_step, 'end_to_end': 1e3 * e2e_s,
                                'host_flatten_and_enumerate_once': 1e3 * host_prep_s},
            'e2e': {'value': A / e2e_s, 'unit': 'plans/s', 'h2d_bytes_per_step': h2d,
                    'd2h_bytes_per_step': int(d2h), 'ms_per_step': 1e3 * e2e_s, 'steps': e2e_steps,
                    'api': 'metis_b200.api.cost_het_cluster(args, gpu_cluster, profile_data, model_config, '
                           'cost_estimator, layer_load_balancer) + len(result) + result.best()',
                    'breakdown_ms': mean_part,
                    'timing': 'wall clock between device synchronisations, max over ranks; includes flattening of the '
                              'profile dicts, host listing of the compositions, H2D, the row kernel, search kernels, sort, D2H; excludes only '
                              'the first two calls (allocation of pinned / device buffers, reused afterwards)'},
            # per timed step: pack_tables, range_sums, het_admit, het_scatter, het_first, het_order, het_chain, het_finalize
            'gpu_launches': 8 * ns.steps,
            'kernel_ms': {'search_kernels_mean': kernel_ms, 'step_mean': ms_per_step,
                          'step_min': min(step_ms), 'step_max': max(step_ms),
                          'note': 'search_kernels = het_admit + het_scatter + het_first + het_chain (CUDA events '
                                  'recorded by the library around those four launches)'},
            'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
                         'frac': achieved / peak, 'traffic': traffic,
                         'peak_source': 'MEASURED_PEAKS.json hbm_gbs (measured)' if 'hbm_gbs' in peaks else 'fallback',
                         'algorithmic_bytes_per_launch': alg_bytes // world,
                         'note': 'S+16 B read per inter-stage plan + 16 B written per costed candidate (SURVEY.md 8d) over '
                                 'the time of the four search kernels (the chain kernel dominates); the path is '
                                 'fp64-latency / instruction-issue bound, not HBM bound'},
            'clocks': sampler.summary() if sampler else None,
            'wall_s_timed_region': wall,
        }
        if world == 1 and not ns.no_cpu:
            arm = CpuArm(ns.workload, A, ns.cpu_sample, 1)
            a, c, t = arm.step(0)
            line['cpu_baseline'] = {'value': a / t, 'unit': 'plans/s', 'cores': arm.cores, 'kind': arm.kind,
                                    'sample': arm.describe(a, c, A, t)}
            arm.close()
        if emit:
            emit_result(line)
    if world > 1:
        dist.barrier()
    del full, probe, dp, flush
    api.release_engines()
    torch.cuda.empty_cache()
    tmp.cleanup()
    return line if rank == 0 else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default=DEFAULT_WORKLOAD)
    ap.add_argument('--cpu-sample', type=int, default=3000, help='plans per host core for cpu_baseline')
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--no-extra', action='store_true', help='skip the configs[3] measurements reported under `extra`')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last timed search computed as DIR/<name>.npy (float64): '
                         'the headline workload only (not the workloads under `extra`); with --workload a,b '
                         'DIR/<workload>/, with several ranks DIR/rank<r>/')
    ns = ap.parse_args()
    if ns.steps < 1:
        ap.error('--steps must be at least 1')
    if ns.dump_outputs and ns.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of the GPU search (--impl ours)')
    # stdout carries exactly one JSON line: libraries that write to fd 1 (NCCL prints its version there when
    # NCCL_DEBUG=VERSION) are sent to stderr for the duration of the run
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)
    if ns.impl == 'reference':
        run_reference_arm(ns)
        return
    # --workload a,b,c (developer use: the scaling table of profiles/) runs the workloads one after the other in
    # this process group and prints one line each; the default invocation prints exactly one line
    names = ns.workload.split(',')
    if names == [DEFAULT_WORKLOAD] and not ns.no_extra:
        # the headline line (BASELINE configs[2]) + the two configs[3] spaces, measured the same way, under `extra`
        # (the 1 -> 8 scaling of the large spaces is where the GPUs pay off)
        line = run_ours(ns, emit=False, dump_dir=ns.dump_outputs)
        extra = {}
        for name in EXTRA_WORKLOADS:
            sub = argparse.Namespace(**vars(ns))
            sub.workload, sub.no_cpu = name, True
            try:
                other = run_ours(sub, emit=False)
            except Exception as exc:                          # noqa: BLE001 - the headline line must still be printed
                extra[name] = {'error': f'{type(exc).__name__}: {exc}'[:200]}
                continue
            if other is not None:
                extra[name] = {'inter_stage_plans': other['config']['inter_stage_plans'], 'value': other['value'],
                               'ms_per_step': other['ms_per_step'], 'steps': other['steps'],
                               'e2e_value': other['e2e']['value'], 'e2e_ms_per_step': other['e2e']['ms_per_step'],
                               'C_costed': other['counters']['C_costed'], 'unit': 'plans/s'}
        if line is not None:
            line['extra'] = extra
            emit_result(line)
    else:
        for name in names:
            ns.workload = name
            dump = ns.dump_outputs
            if dump and len(names) > 1:
                dump = os.path.join(dump, name)
            run_ours(ns, dump_dir=dump)
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        dist.destroy_process_group()


_RESULT_FD = None


def emit_result(line):
    data = (json.dumps(line) + '\n').encode()
    sys.stdout.flush()
    if _RESULT_FD is None:
        os.write(1, data)
    else:
        os.write(_RESULT_FD, data)


if __name__ == '__main__':
    main()
