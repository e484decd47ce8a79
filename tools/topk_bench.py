#!/usr/bin/env python3
"""Top-k plan search against the whole list: one JSON line per measurement.

  python tools/topk_bench.py [--workloads ...] [--ks 1 10 1000] [--steps 5] [--warmup 2] [--out FILE]
  torchrun --nproc-per-node 8 tools/topk_bench.py ...

kind=hardware  the card's name and power limit (nvidia-smi, read only), read in the same run
kind=e2e       seconds per call from host inputs, synchronised, after warm-up calls, the two ways a caller gets the k best
               plans: api.best_het_plans(k) and api.cost_het_cluster(...).ranked(k) (k tuples built in both); the calls
               alternate step by step and the two answers are checked equal
kind=kernel    device time (CUDA events over --launches launches) of metis_select_records(k) against
               metis_sort_records(RANKED) on the same device-resident records (the rank's whole candidate list)
Under torchrun every rank runs the same calls; e2e times are the maximum over the ranks, kernel times rank 0's.
"""
import argparse
import itertools
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def hardware(local: int):
    import torch
    q = subprocess.run(['nvidia-smi', '-i', str(local), '--query-gpu=name,power.limit,clocks.max.sm',
                        '--format=csv,noheader'], capture_output=True, text=True)
    return {'kind': 'hardware', 'torch_device_name': torch.cuda.get_device_name(local),
            'nvidia_smi': q.stdout.strip() if q.returncode == 0 else f'unavailable: {q.stderr.strip()}'}


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('--workloads', nargs='+', default=['c3_homo64_mpl6', 'c4_het128', 'c4_het128_mpl6'])
    ap.add_argument('--ks', nargs='+', type=int, default=[1, 10, 1000])
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--launches', type=int, default=20)
    ap.add_argument('--out', default=None, help='also append the JSON lines to this file (rank 0)')
    ns = ap.parse_args(argv)
    if ns.steps < 1 or ns.warmup < 1 or ns.launches < 1:
        raise SystemExit('--steps, --warmup and --launches must be at least 1')

    import torch
    import torch.distributed as dist
    from metis_b200 import api, native, search
    from metis_b200.arguments import parse_args
    from metis_b200.data_loader import ProfileDataLoader
    from metis_b200.gpu_cluster import GPUCluster
    from metis_b200.utils import ModelConfig
    from metis_b200.workloads import WORKLOADS, materialize, profile_file_order

    if not torch.cuda.is_available():
        raise SystemExit('topk_bench.py needs a CUDA device')
    native.load_library()
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device(f'cuda:{local}')
    if world > 1 and not dist.is_initialized():
        dist.init_process_group('nccl', device_id=dev)

    def emit(obj):
        if rank == 0:
            line = json.dumps(dict(obj, world=world))
            print(line, flush=True)
            if ns.out:
                with open(ns.out, 'a') as fh:
                    fh.write(line + '\n')

    def worst(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    emit(hardware(local))
    for name in ns.workloads:
        w = WORKLOADS[name]
        tmp = tempfile.TemporaryDirectory()
        materialize(w, tmp.name)
        args = parse_args(w.cli_args(tmp.name))
        cluster = GPUCluster(args.hostfile_path, args.clusterfile_path)
        profile, _ = ProfileDataLoader(args.profile_data_path, profile_file_order(w)).load_profile_data_all()
        cfg = ModelConfig(model_name=args.model_name, num_layers=args.num_layers, sequence_length=args.sequence_length,
                          vocab_size=args.vocab_size, hidden_size=args.hidden_size,
                          attention_head_size=args.attention_head_size)
        volume = api.GPTActivationAndParam(cfg, profile['model']['parameters'])
        call = (args, cluster, profile, cfg, api.HeteroCostEstimator(profile, cfg, volume, cluster),
                api.LayerLoadBalancer(cluster, profile, cfg, args.gbs))
        seqs = list(itertools.permutations(w.device_types()))

        # ---- e2e: the two ways to the k best plans, alternating --------------------------------------------------
        for k in ns.ks:
            def top_k():
                return list(api.best_het_plans(*call, k, node_sequences=seqs, device=dev))

            def whole_then_ranked():
                return api.cost_het_cluster(*call, node_sequences=seqs, device=dev).ranked(k)
            wall = {'best_het_plans': [], 'cost_het_cluster_ranked': []}
            answers = {}
            for i in range(ns.warmup + ns.steps):
                for label, fn in (('best_het_plans', top_k), ('cost_het_cluster_ranked', whole_then_ranked)):
                    if world > 1:
                        dist.barrier()
                    torch.cuda.synchronize(dev)
                    t0 = time.perf_counter()
                    answers[label] = fn()
                    torch.cuda.synchronize(dev)
                    if i >= ns.warmup:
                        wall[label].append(time.perf_counter() - t0)
            same = answers['best_het_plans'] == answers['cost_het_cluster_ranked']
            if not same:
                raise SystemExit(f'{name} k={k}: best_het_plans differs from cost_het_cluster(...).ranked(k)')
            res = {f'{label}_ms': 1e3 * worst(statistics.mean(v)) for label, v in wall.items()}
            res.update({f'{label}_min_ms': 1e3 * worst(min(v)) for label, v in wall.items()})
            emit(dict(kind='e2e', workload=name, k=k, steps=ns.steps, answers_equal=same, **res))

        # ---- kernels on this rank's device-resident records -------------------------------------------------------
        problem, space, _ = api.het_problem(args, cluster, profile, cfg, call[5], seqs, device_rows=True)
        dp = search.DeviceProblem(problem, space, dev)
        searcher = search.HetSearcher(dp, rank, world, want_records=True, want_detail=False)
        out = searcher.run()
        n = out.summary['num_records']
        recs = out.records_dev.clone()
        s = torch.cuda.current_stream(dev)

        def timed(fn):
            fn()
            s.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(s)
            for _ in range(ns.launches):
                fn()
            b.record(s)
            s.synchronize()
            return a.elapsed_time(b) / ns.launches
        sort_buf = recs.clone()
        sort_ms = timed(lambda: searcher.sort_records(n, native.SORT_RANKED, s, buf=sort_buf))
        for k in ns.ks:
            top, _ = searcher.select_records(recs, n, k, s)
            want = sort_buf[:2 * min(k, n)]
            assert torch.equal(top, want), f'{name} k={k}: selection differs from the sort'
            sel_ms = timed(lambda: searcher.select_records(recs, n, k, s))
            emit(dict(kind='kernel', workload=name, rank=rank, records=n, record_bytes=16 * n, k=k,
                      select_ms=sel_ms, sort_ranked_ms=sort_ms, launches=ns.launches))
        del dp, searcher, out, recs, sort_buf
        api.release_engines()
        tmp.cleanup()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
