#!/usr/bin/env python3
"""Small searches for compute-sanitizer (memcheck / racecheck): forces both schedules (bulk round + chains, chains only)."""
import itertools, os, sys, tempfile
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from metis_b200 import flatten, search
from metis_b200.data_loader import ProfileDataLoader
from metis_b200.gpu_cluster import GPUCluster
from metis_b200.utils import ModelConfig
from metis_b200.workloads import WORKLOADS, materialize, profile_file_order

for name in sys.argv[1:] or ['c2_v100', 'mix32']:
    w = WORKLOADS[name]
    tmp = tempfile.mkdtemp(); materialize(w, tmp)
    cluster = GPUCluster(tmp + '/hostfile', tmp + '/clusterfile.json')
    profile, _ = ProfileDataLoader(tmp + '/profile', profile_file_order(w)).load_profile_data_all()
    cfg = ModelConfig('SYN', w.num_layers, w.sequence_length, w.vocab_size, w.hidden_size, 32)
    seqs = list(itertools.permutations(w.device_types()))
    problem = flatten.build_problem(profile, cluster, cfg, w.gbs, w.max_tp, w.max_bs, seqs)
    # rows written by the GPU (het_rows_kernel) so that kernel runs under the sanitizer too
    space = flatten.build_plan_space(len(seqs), cluster.get_total_num_devices(), w.gbs, w.num_layers, w.variance, w.max_permute_len,
                                     device_rows=True)
    dp = search.DeviceProblem(problem, space, 'cuda:0')
    for coop in (1, 2 ** 31 - 1):
        s = search.HetSearcher(dp, want_records=True, want_detail=True, want_ranking=True)
        s.shard.reserved = coop
        out = s.run()
        print(name, 'coop factor', coop, out.summary['num_records'], out.best[:3], 'ranked first', int(out.rank_order[0]))
    # top-k path: the local selection on the search's unordered records, then a merge selection over two lists
    import torch
    t = search.HetSearcher(dp, want_records=True, want_detail=False)
    top = t.run_top(10)
    both = torch.cat([top.records_dev, out.records_dev]).contiguous()
    merged, idx = t.select_records(both, both.numel() // 2, 10, torch.cuda.current_stream(), want_idx=True)
    picks = merged.cpu().numpy().view('u1').view(search.native.RECORD_DTYPE)
    rows = t.detail_for(picks)
    torch.cuda.synchronize()
    print(name, 'top-k', top.records_dev.numel() // 2, 'merged first', picks[0], 'from', int(idx[0]), rows.shape)
