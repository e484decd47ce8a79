"""Top-k plan search on the GPU: metis_select_records against numpy's stable sort, and api.best_het_plans against
cost_het_cluster(...).ranked(k), the golden candidates, the fatal cases, the corrections, the CLI transcript and two
ranks over NCCL."""
import ctypes as C
import gzip
import json
import os
import pickle
import socket
import subprocess
import sys

import numpy as np
import pytest

from conftest import C1_DIR, GOLDEN, REPO, golden_best, load_golden

pytestmark = pytest.mark.gpu

C1_ARGV = ['--model_name', 'GPT', '--model_size', '1.5B', '--num_layers', '10', '--gbs', '128',
           '--max_profiled_tp_degree', '4', '--max_profiled_batch_size', '4', '--min_group_scale_variance', '1',
           '--max_permute_len', '4', '--hidden_size', '4096', '--sequence_length', '1024', '--vocab_size', '51200',
           '--attention_head_size', '32', '--hostfile_path', os.path.join(C1_DIR, 'hostfile'),
           '--clusterfile_path', os.path.join(C1_DIR, 'clusterfile.json'),
           '--profile_data_path', os.path.join(C1_DIR, 'profile_data_samples')]


def _gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from metis_b200 import native
    native.load_library()
    return torch


def _select_on_device(rec_np, k):
    import torch
    from metis_b200 import native
    lib = native.load_library()
    n = len(rec_np)
    m = min(k, n)
    raw = torch.from_numpy(rec_np.view(np.uint8).reshape(-1).copy()).cuda() if n else torch.zeros(16, dtype=torch.uint8).cuda()
    out = torch.full((max(m, 1) * 16,), 0xAB, dtype=torch.uint8, device='cuda')
    idx = torch.full((max(m, 1),), -1, dtype=torch.int32, device='cuda')
    ws = torch.empty(int(lib.metis_select_workspace_bytes(n, k)), dtype=torch.uint8, device='cuda')
    rc = lib.metis_select_records(C.c_void_p(raw.data_ptr()), C.c_int64(n), C.c_int64(k), C.c_void_p(out.data_ptr()),
                                  C.c_void_p(idx.data_ptr()), C.c_void_p(ws.data_ptr()), C.c_int64(ws.numel()),
                                  C.c_void_p(torch.cuda.current_stream().cuda_stream))
    native.check(rc, 'metis_select_records')
    torch.cuda.synchronize()
    assert (raw.cpu().numpy()[:n * 16] == rec_np.view(np.uint8).reshape(-1)).all(), 'the input was modified'
    return out.cpu().numpy()[:m * 16].view(native.RECORD_DTYPE), idx.cpu().numpy()[:m].view(np.uint32)


@pytest.mark.parametrize('n', [0, 1, 31, 32, 33, 1000, 100003, 3_000_000])
def test_selection_is_the_head_of_the_stable_ranked_sort(n):
    """metis_select_records against rec[np.lexsort((step, ordinal, cost))][:k]: repeated costs, inf, 1e300, the
    smallest subnormal, negative costs, costs one ulp apart, ordinals up to 2^32, steps up to 2^16, equal keys (kept
    in input order), and a case where every cost is equal so that only (ordinal, step) decides."""
    _gpu()
    from metis_b200 import native
    rng = np.random.default_rng(n + 11)
    pool = np.concatenate([rng.uniform(-1e3, 1e6, 40), [np.inf, 1e300, 5e-324, 1.0, 1.0000000000000002, -7.5,
                                                        -1.0000000000000002, -1.0]])
    cases = []
    for equal_costs in (False, True):
        rec = np.zeros(n, dtype=native.RECORD_DTYPE)
        rec['cost'] = 621.8881853975784 if equal_costs else rng.choice(pool, n)
        rec['ordinal'] = rng.integers(0, 2 ** 32, n, dtype=np.uint64).astype(np.uint32) if n % 2 else rng.integers(0, 5000, n)
        rec['step'] = rng.integers(0, 2 ** 16, n) if n % 3 == 0 else rng.integers(0, 19, n)
        rec['num_repartition'] = rng.integers(1, 4, n)
        rec['num_stage'] = rng.integers(1, 129, n)
        cases.append(rec)
    for rec in cases:
        want = np.lexsort((rec['step'], rec['ordinal'], rec['cost']))
        for k in sorted({0, 1, 7, 4096, max(n - 1, 0), n, n + 5}):
            got, idx = _select_on_device(rec, k)
            m = min(k, n)
            assert len(got) == m
            assert (idx == want[:m]).all(), (n, k)
            assert (got.view(np.uint8) == rec[want[:m]].view(np.uint8)).all(), (n, k)


def test_selection_rejects_bad_arguments():
    _gpu()
    from metis_b200 import native
    lib = native.load_library()
    assert lib.metis_select_workspace_bytes(-1, 3) < 0 and lib.metis_select_workspace_bytes(3, -1) < 0
    ws = 256                                                 # rejected before the workspace is touched
    assert lib.metis_select_records(None, 2 ** 32, 5, None, None, ws, 16, None) == -2
    assert lib.metis_select_records(None, 10, -1, None, None, ws, 16, None) == -2
    assert lib.metis_select_records(None, 0, 5, None, None, ws, lib.metis_select_workspace_bytes(0, 5), None) == 0


# ---------------------------------------------------------------------------------------------------------------
# api.best_het_plans
# ---------------------------------------------------------------------------------------------------------------
def _api_inputs(name, workload_dir):
    from metis_b200 import api
    from metis_b200.arguments import parse_args
    from metis_b200.data_loader import ProfileDataLoader
    from metis_b200.gpu_cluster import GPUCluster
    from metis_b200.utils import ModelConfig
    if name == 'c1':
        meta, arr = load_golden('c1_het')
        args = parse_args(C1_ARGV)
    else:
        meta, arr = load_golden(name)
        w, root, _ = workload_dir(name)
        args = parse_args(w.cli_args(root))
    cluster = GPUCluster(args.hostfile_path, args.clusterfile_path)
    profile, _ = ProfileDataLoader(args.profile_data_path, meta['file_order']).load_profile_data_all()
    cfg = ModelConfig(model_name='t', num_layers=args.num_layers, sequence_length=args.sequence_length,
                      vocab_size=args.vocab_size, hidden_size=args.hidden_size, attention_head_size=32)
    volume = api.GPTActivationAndParam(cfg, profile['model']['parameters'])
    est = api.HeteroCostEstimator(profile, cfg, volume, cluster)
    llb = api.LayerLoadBalancer(cluster, profile, cfg, args.gbs)
    seqs = [tuple(s) for s in meta['node_sequences']]
    return meta, arr, (args, cluster, profile, cfg, est, llb), seqs


@pytest.mark.parametrize('name', ['c1', 'mix32', 'het32_tight', 'c2_het16', 'sweep_n16_t2_v0', 'c3_homo64_mpl4'])
def test_best_het_plans_is_the_head_of_the_ranked_list(name, workload_dir):
    _gpu()
    from metis_b200 import api
    meta, arr, call, seqs = _api_inputs(name, workload_dir)
    full = api.cost_het_cluster(*call, node_sequences=seqs, device='cuda:0')
    ranked = full.ranked()
    c = meta['counters']
    C_ = len(full)
    assert C_ == c['C']
    gold_order = np.lexsort((arr['step'], arr['ordinal'], arr['cost'])) if 'rows' not in arr else None
    for k in (1, 10, C_, C_ + 3):
        top = api.best_het_plans(*call, k, node_sequences=seqs, device='cuda:0')
        assert isinstance(top, api.HetTopResult) and len(top) == min(k, C_)
        assert list(top) == ranked[:k] == full.ranked(k), (name, k)
        assert top == ranked[:k] and top[0] == full.best() and top[-1] == ranked[min(k, C_) - 1]
        assert top[0][6] == golden_best(meta, arr)[0]
        assert (top.costs.view(np.uint64) == np.array([r[6] for r in ranked[:k]]).view(np.uint64)).all()
        if gold_order is not None:
            assert (top.costs.view(np.uint64) == arr['cost'][gold_order[:k]].view(np.uint64)).all()
        s = top.summary
        assert (s['num_plans'], s['num_partition_calls'], s['num_balancer_runs'], s['num_records'], s['num_keyerror']) \
            == (c['A'], c['B'], c['runs'], c['C'], c['keyerr']), (name, k, s)
        assert s['corrected'] == () and s['fatal_ordinal'] == 2 ** 64 - 1
    assert list(api.best_het_plans(*call, 0, node_sequences=seqs, device='cuda:0')) == []
    with pytest.raises(ValueError, match='k must be >= 0'):
        api.best_het_plans(*call, -1, node_sequences=seqs, device='cuda:0')
    with pytest.raises(ValueError, match='unknown corrections'):
        api.best_het_plans(*call, 3, node_sequences=seqs, device='cuda:0', corrected=('Q9',))


def test_best_het_plans_raises_like_cost_het_cluster(workload_dir):
    _gpu()
    from metis_b200 import api
    for name, exc in (('fatal_gbs96', KeyError), ('q10_small_first', IndexError)):
        meta, _arr, call, seqs = _api_inputs(name, workload_dir)
        with pytest.raises(exc) as want:
            api.cost_het_cluster(*call, node_sequences=seqs, device='cuda:0')
        with pytest.raises(exc) as got:
            api.best_het_plans(*call, 5, node_sequences=seqs, device='cuda:0')
        assert str(got.value) == str(want.value) == meta['fatal'][2]


def test_best_het_plans_with_a_correction(workload_dir):
    _gpu()
    from metis_b200 import api
    _meta, _arr, call, seqs = _api_inputs('mix32', workload_dir)
    full = api.cost_het_cluster(*call, node_sequences=seqs, device='cuda:0', corrected=('Q5',))
    ranked = full.ranked()
    for k in (1, 17, len(full) + 1):
        top = api.best_het_plans(*call, k, node_sequences=seqs, device='cuda:0', corrected=('Q5',))
        assert list(top) == ranked[:k] and top.summary['corrected'] == ('Q5',)
        assert top.summary['num_records'] == full.summary['num_records']


def test_interleaved_calls_on_different_problems(workload_dir):
    """The engine cache serves both functions: alternating problems and functions changes no answer."""
    _gpu()
    from metis_b200 import api
    inputs = {name: _api_inputs(name, workload_dir) for name in ('mix32', 'c2_het16')}
    alone = {}
    for name, (_m, _a, call, seqs) in inputs.items():
        api.release_engines()
        full = api.cost_het_cluster(*call, node_sequences=seqs, device='cuda:0')
        alone[name] = (list(full), full.ranked()[:25])
    api.release_engines()
    for name in ('mix32', 'c2_het16', 'mix32', 'c2_het16', 'mix32'):
        _m, _a, call, seqs = inputs[name]
        top = api.best_het_plans(*call, 25, node_sequences=seqs, device='cuda:0')
        full = api.cost_het_cluster(*call, node_sequences=seqs, device='cuda:0')
        assert list(top) == alone[name][1], name
        assert list(full) == alone[name][0], name
        again = api.best_het_plans(*call, 25, node_sequences=seqs, device='cuda:0')
        assert list(again) == alone[name][1] and list(top) == alone[name][1], name


def test_ranked_k_through_the_selection(workload_dir):
    """HetSearchResult.ranked(k) before the whole ranking exists uses the device selection: same list as ranked()[:k];
    afterwards it slices the full ranking."""
    _gpu()
    from metis_b200 import api
    _meta, _arr, call, seqs = _api_inputs('c3_homo64_mpl4', workload_dir)
    res = api.cost_het_cluster(*call, node_sequences=seqs, device='cuda:0')
    n = len(res)
    got = {k: res.ranked(k) for k in (0, 1, 2, 10, 1000, n - 1)}
    assert res.rank_order is None                            # no full sort has run
    full = res.ranked()
    for k, v in got.items():
        assert v == full[:k], k
    assert res.ranked(n + 3) == full and res.ranked(-2) == full[:-2]


@pytest.mark.parametrize('name,top_k', [('c1', 3), ('c2_het16', 10)])
def test_cli_top_k_stdout_is_the_reference_transcript_cut(name, top_k, workload_dir, capsys, monkeypatch):
    """METIS_TOP_K=N with METIS_VERBOSE=1: the reference's whole stdout with the ranked table cut after N rows
    (`search_time:` masked); `len(costs):` still counts every candidate."""
    _gpu()
    import cost_het_cluster as cli
    from metis_b200.utils import DeviceType
    meta = json.load(open(os.path.join(GOLDEN, f'transcript_{name}.json')))
    gold = gzip.open(os.path.join(GOLDEN, f'transcript_{name}.txt.gz'), 'rt').read().split('\n')
    header = gold.index('rank, cost, node_sequence, device_groups, strategies(dp_deg, tp_deg), batches(number of batch), '
                        'layer_partition')
    assert header + 1 + top_k < len(gold) - 1
    want = gold[:header + 1 + top_k] + ['']
    if name == 'c1':
        argv = C1_ARGV
    else:
        w, root, digest = workload_dir(name)
        assert digest == meta['inputs_sha256']
        argv = w.cli_args(root)
    monkeypatch.setenv('METIS_VERBOSE', '1')
    monkeypatch.setenv('METIS_TOP_K', str(top_k))
    seqs = [tuple(DeviceType[t] for t in seq) for seq in meta['node_sequences']]
    capsys.readouterr()
    cli.main(argv, node_sequences=seqs, file_order=meta['file_order'])
    ours = capsys.readouterr().out.split('\n')
    ours = ['search_time: <masked>' if ln.startswith('search_time: ') else ln for ln in ours]
    assert len(ours) == len(want)
    for i, (a, b) in enumerate(zip(ours, want)):
        assert a == b, f'line {i + 1} differs'


TWO_RANKS = r'''
import os, pickle, sys
sys.path.insert(0, os.environ['REPO']); sys.path.insert(0, os.path.join(os.environ['REPO'], 'tests'))
import torch, torch.distributed as dist
rank = int(os.environ['RANK'])
torch.cuda.set_device(rank)
dist.init_process_group('nccl', init_method='tcp://127.0.0.1:' + os.environ['PORT'], rank=rank, world_size=2,
                        device_id=torch.device(f'cuda:{rank}'))
from metis_b200 import api
call, seqs, ks = pickle.load(open(os.environ['INPUTS'], 'rb'))
out = {}
for k in ks:
    top = api.best_het_plans(*call, k, node_sequences=seqs, device=f'cuda:{rank}')
    out[k] = (list(top), {key: top.summary[key] for key in ('num_records', 'num_partition_calls', 'num_balancer_runs')})
pickle.dump(out, open(os.environ['OUT'], 'wb'))
dist.barrier(); dist.destroy_process_group()
'''


def test_two_ranks_return_the_single_gpu_top_k(workload_dir, tmp_path):
    torch = _gpu()
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    from metis_b200 import api
    _meta, _arr, call, seqs = _api_inputs('c3_homo64_mpl4', workload_dir)
    C_ = _meta['counters']['C']
    ks = [1, 10, 1000, C_ + 3]
    want = {k: list(api.best_het_plans(*call, k, node_sequences=seqs, device='cuda:0')) for k in ks}
    full = api.cost_het_cluster(*call, node_sequences=seqs, device='cuda:0')
    inputs = tmp_path / 'inputs.pkl'
    pickle.dump((call, seqs, ks), open(inputs, 'wb'))
    script = tmp_path / 'worker.py'
    script.write_text(TWO_RANKS)
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    procs = []
    for rank in range(2):
        env = dict(os.environ, REPO=REPO, RANK=str(rank), PORT=str(port), INPUTS=str(inputs),
                   OUT=str(tmp_path / f'rank{rank}.pkl'))
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=600)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), '\n'.join(outs)
    for rank in range(2):
        got = pickle.load(open(tmp_path / f'rank{rank}.pkl', 'rb'))
        for k in ks:
            assert got[k][0] == want[k], (rank, k)
            assert got[k][1] == {key: full.summary[key] for key in got[k][1]}, (rank, k)
