"""CPU tests of the top-k path: the multi-rank merge of best_het_plans (world 2 over gloo, the device selection
replaced by numpy) and the parsing of METIS_TOP_K."""
import os
import re
import socket
import subprocess
import sys

import pytest

from conftest import REPO, load_golden

WORKER = r'''
import os, sys
sys.path.insert(0, os.environ['REPO']); sys.path.insert(0, os.path.join(os.environ['REPO'], 'tests'))
import torch, torch.distributed as dist
dist.init_process_group('gloo', init_method='tcp://127.0.0.1:' + os.environ['PORT'],
                        rank=int(os.environ['RANK']), world_size=2)
import numpy as np
import hostsim_util as hs
from conftest import load_golden
from metis_b200 import flatten, native, search
from metis_b200.workloads import WORKLOADS, materialize
import tempfile

def np_select(records, k):
    """numpy stand-in of metis_select_records: the first k of the stable (cost, ordinal, step) order."""
    rec = records.numpy().view(np.uint8).view(native.RECORD_DTYPE)
    order = np.lexsort((rec['step'], rec['ordinal'], rec['cost']))[:k]
    return torch.from_numpy(np.ascontiguousarray(rec[order]).view(np.int64).copy())

meta, arr = load_golden('c2_v100')
w = WORKLOADS['c2_v100']
root = tempfile.mkdtemp(); materialize(w, root)
cluster, profile, _, cfg = hs.load_inputs(root, 'profile', meta['file_order'], w.num_layers, w.hidden_size, w.sequence_length, w.vocab_size)
seqs = [tuple(s) for s in meta['node_sequences']]
problem = flatten.build_problem(profile, cluster, cfg, w.gbs, w.max_tp, w.max_bs, seqs)
space = flatten.build_plan_space(len(seqs), 16, w.gbs, w.num_layers, w.variance, w.max_permute_len)
rank = dist.get_rank()
rec, _det, sm = hs.host_het_search(problem, space, rank=rank, world=2, tile=64, want_detail=False)   # shard: test shim
summary = dict(num_records=int(sm.num_records), num_partition_calls=int(sm.num_partition_calls),
               num_balancer_runs=int(sm.num_balancer_runs), num_keyerror=int(sm.num_keyerror),
               fatal_ordinal=int(sm.fatal_ordinal), fatal_code=int(sm.fatal_code), fatal_aux=int(sm.fatal_aux))
local_best = (sm.best.cost, sm.best.ordinal, sm.best.step, sm.best.num_repartition, sm.best.num_stage)
c = meta['counters']
assert 0 < sm.num_records < c['C']
order = np.lexsort((arr['step'], arr['ordinal'], arr['cost']))
for k in (1, 10, 300, c["C"], c["C"] + 3):          # 300: more than one shard holds
    local_top = np_select(torch.from_numpy(np.ascontiguousarray(rec).view(np.int64).copy()), k)
    merged, best, top = search.global_top(summary, local_best, local_top, k, 'cpu', select=np_select)
    got = top.numpy().view(np.uint8).view(native.RECORD_DTYPE)
    want = order[:k]
    assert len(got) == min(k, c['C'])
    assert (got['ordinal'] == arr['ordinal'][want]).all() and (got['step'] == arr['step'][want]).all()
    assert (got['cost'].view(np.uint64) == arr['cost'][want].view(np.uint64)).all()
    assert (got['num_repartition'] == arr['nrep'][want]).all() and (got['num_stage'] == arr['nstage'][want]).all()
    assert (merged['num_records'], merged['num_partition_calls'], merged['num_balancer_runs']) == (c['C'], c['B'], c['runs'])
    assert merged['fatal_ordinal'] == 2 ** 64 - 1 and best[:3] == (got['cost'][0], got['ordinal'][0], got['step'][0])
# one rank's failure makes both ranks raise: its own exception there, a named error on the other
try:
    search.global_top(summary, local_best, None if rank == 1 else local_top, 5, 'cpu',
                      failure=RuntimeError('search failed on rank 1') if rank == 1 else None, select=np_select)
except RuntimeError as exc:
    assert ('search failed on rank 1' in str(exc)) if rank == 1 else isinstance(exc, native.MetisNativeError), exc
else:
    raise AssertionError('no rank may return after another rank failed')
# a fatal plan on one rank: every rank sees the lowest fatal ordinal and no records are exchanged
fatal = dict(summary, fatal_ordinal=40 + rank, fatal_code=1 + 2 * rank, fatal_aux=(1 << 16) | 3)
merged, _, top = search.global_top(fatal, local_best, local_top, 5, 'cpu', select=np_select)
assert top is None and (merged['fatal_ordinal'], merged['fatal_code']) == (40, 1)
dist.barrier(); dist.destroy_process_group()
print('rank', rank, 'ok')
'''


def test_two_rank_top_k_merge_gloo(tmp_path):
    """world 2 over gloo: each rank's shard from the host build of the search, its local k best, then
    search.global_top (the product's exchange and merge, with numpy in place of the device selection) gives the global
    k best of the golden c2_v100 on both ranks, and spreads a rank's error or fatal plan to both."""
    load_golden('c2_v100')
    import hostsim_util
    hostsim_util.hostsim()                      # build the test shim once, before the ranks start
    script = tmp_path / 'worker.py'
    script.write_text(WORKER)
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    procs = []
    for rank in range(2):
        env = dict(os.environ, REPO=REPO, RANK=str(rank), PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=300)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), '\n'.join(outs)


@pytest.mark.parametrize('raw,want', [(None, None), ('', None), ('  ', None), ('0', 0), ('7', 7), (' 12 ', 12),
                                      ('1000000', 1000000)])
def test_metis_top_k_values(raw, want):
    from cost_het_cluster import top_k_from_env
    assert top_k_from_env({} if raw is None else {'METIS_TOP_K': raw}) == want


@pytest.mark.parametrize('raw', ['-1', '-0x1', 'ten', '1.5', '1e3', '0x10', '3 4'])
def test_metis_top_k_refuses_anything_but_a_count(raw):
    from cost_het_cluster import top_k_from_env
    with pytest.raises(ValueError, match=re.escape(f'METIS_TOP_K must be a non-negative integer, got {raw!r}')):
        top_k_from_env({'METIS_TOP_K': raw})
