"""Host-side mirror of the reference's interface for the plan-search path.

Same class / function names, argument meaning and error behaviour as the reference, so that
``cost_het_cluster.py`` / ``cost_homo_cluster.py`` read like the originals; the objects are thin
holders of inputs - every evaluation happens on the GPU (metis_b200.search).

  reference symbol                                   here
  -------------------------------------------------  -------------------------------------------
  model/activation_parameter.py GPTActivationAndParam  GPTActivationAndParam
  model/cost_estimator.py HeteroCostEstimator           HeteroCostEstimator   (holder)
  model/cost_estimator.py HomoCostEstimator             HomoCostEstimator     (holder)
  model/load_balancer.py LayerLoadBalancer              LayerLoadBalancer     (holder + norm_layer_duration)
  search_space/plan.py UniformPlan / InterStagePlan     same dataclasses
  search_space/plan.py UniformPlanGenerator             UniformPlanGenerator  (host iterator)
  search_space/plan.py InterStagePlanGenerator          InterStagePlanGenerator (iterator over the plan space)
  cost_het_cluster.py cost_het_cluster()                cost_het_cluster()    -> GPU
  cost_het_cluster(...) then sorted(...)[:k]            best_het_plans(..., k) -> GPU (no whole list)
  cost_homo_cluster.py cost_homo_cluster()              cost_homo_cluster()   -> GPU
"""
from __future__ import annotations

import argparse
import operator
import time
from dataclasses import dataclass
from itertools import permutations
from collections.abc import Sequence
from typing import Dict, Iterator, List, Optional, Tuple

import numpy as np

from . import flatten, native
from .utils import DeviceType, ModelConfig


@dataclass
class UniformPlan:
    dp: int
    pp: int
    tp: int
    mbs: int
    gbs: int


@dataclass
class InterStagePlan:
    ns_idx: int
    node_sequence: List[DeviceType]
    dg_idx: int
    device_groups: List[int]
    num_stage: int
    batches: int
    gbs: int


class GPTActivationAndParam:
    """model/activation_parameter.py:5-51 (only the three per-layer sizes reach the kernels)."""

    def __init__(self, model_config: ModelConfig, model_params):
        self.hidden_size = model_config.hidden_size
        self.sequence_length = model_config.sequence_length
        self.num_layers = model_config.num_layers
        self.vocab_size = model_config.vocab_size
        self.attention_head_size = model_config.attention_head_size
        self.input_params = float(model_params[0])
        self.output_params = float(model_params[-1])
        self.transformer_params = float(model_params[1])

    def get_num_layers(self):
        return self.num_layers


class _Estimator:
    def __init__(self, profile_data: Dict, model_config: ModelConfig, model_volume, gpu_cluster):
        self.profile_data = profile_data
        self.model_config = model_config
        self.model_volume = model_volume
        self.gpu_cluster = gpu_cluster


class HeteroCostEstimator(_Estimator):
    """Inputs of model/cost_estimator.py:141-244; evaluated by het_search_kernel."""


class HomoCostEstimator(_Estimator):
    """Inputs of model/cost_estimator.py:83-138; evaluated by homo_cost_kernel."""


class LayerLoadBalancer:
    """Inputs of model/load_balancer.py:14-144; ``norm_layer_duration`` is computed at construction
    like the reference (:20-27) and raises the same KeyError when tp1_bs1 is not profiled."""

    def __init__(self, gpu_cluster, profile_data: Dict, model_config, gbs: int):
        self.gpu_cluster = gpu_cluster
        self.profile_data = profile_data
        self.model_config = model_config
        self.gbs = gbs
        self.norm_layer_duration = flatten.norm_layer_duration(profile_data)


class UniformPlanGenerator:
    """search_space/plan.py:40-97; like the reference it re-yields ONE mutated object."""

    def __init__(self, num_devices: int, max_tp: int, max_gbs: int):
        self.num_devices = num_devices
        self.max_tp = max_tp
        self.max_gbs = max_gbs
        self.curr = UniformPlan(dp=num_devices, pp=1, tp=1, gbs=num_devices, mbs=0)

    def __iter__(self):
        return self

    def _advance_parallelism(self) -> bool:
        p = self.curr
        while True:
            if p.tp == self.max_tp and p.pp == self.num_devices:
                return False
            if p.tp == self.max_tp:
                p.pp += 1
                p.dp = self.num_devices // p.pp
                p.tp = self.num_devices // p.dp // p.pp
            else:
                p.tp += 1
                p.dp = self.num_devices // p.tp // p.pp
            if p.dp * p.pp * p.tp == self.num_devices:
                return True

    def __next__(self) -> UniformPlan:
        p = self.curr
        p.mbs += 1
        while p.gbs % p.mbs > 0 and p.mbs <= p.gbs:
            p.mbs += 1
        if p.mbs * p.dp > p.gbs:
            p.mbs = 1
            p.gbs += 1
            while self.max_gbs % p.gbs > 0 and p.gbs <= self.max_gbs:
                p.gbs += 1
        if p.gbs > self.max_gbs:
            p.mbs = 1
            if not self._advance_parallelism():
                raise StopIteration
            p.gbs = p.dp
        return p


class InterStagePlanGenerator:
    """search_space/plan.py:100-175 as an iterator over the enumerated plan space (quirk Q1 included).
    Each item is a fresh InterStagePlan (the reference mutates one object)."""

    def __init__(self, device_types: set, num_devices: int, gbs: int, num_layers: int, variance: float = 0.5,
                 max_permute_len: int = 4):
        self.node_sequences = list(permutations(device_types))
        self.gbs = gbs
        self.space = flatten.build_plan_space(len(self.node_sequences), num_devices, gbs, num_layers, variance,
                                              max_permute_len)

    def __iter__(self) -> Iterator[InterStagePlan]:
        for ordinal in range(self.space.num_plans):
            ns, label, row, batches, codes = self.space.locate(ordinal)
            yield InterStagePlan(ns_idx=ns, node_sequence=self.node_sequences[ns], dg_idx=row,
                                 device_groups=[1 << int(c) for c in codes], num_stage=label, batches=batches,
                                 gbs=self.gbs)


class _TupleSequence(Sequence):
    """A read-only sequence of the reference's 7-tuples
    ``(node_sequence, device_groups, strategies, batches, layer_partition, num_repartition, cost)`` whose tuples are
    built from ``candidates`` (search.Candidates) when they are asked for.  ``len()``, indexing, slicing, iteration,
    ``sorted(result, key=...)`` and comparison with a list behave like a list's."""

    def __init__(self, candidates, summary: Dict[str, int], timings: Optional[Dict[str, float]] = None):
        self.candidates = candidates
        self.summary = summary
        self.timings = timings or {}

    def __len__(self) -> int:
        return len(self.candidates)

    def __getitem__(self, i):
        n = len(self)
        if isinstance(i, slice):
            return self.candidates.tuples(np.arange(n)[i])
        i = int(i)
        if i < 0:
            i += n
        if not 0 <= i < n:
            raise IndexError('list index out of range')
        return self.candidates.tuples([i])[0]

    def __iter__(self) -> Iterator[Tuple]:
        n = len(self)
        for lo in range(0, n, 8192):
            yield from self.candidates.tuples(np.arange(lo, min(n, lo + 8192)))

    def __eq__(self, other) -> bool:
        if not isinstance(other, (list, tuple, Sequence)) or len(other) != len(self):
            return False
        return all(a == b for a, b in zip(self, other))

    __hash__ = None

    @property
    def costs(self) -> np.ndarray:
        """fp64 cost of every entry, in the sequence's order (no tuples built)."""
        return self.candidates.cost


class HetSearchResult(_TupleSequence):
    """What cost_het_cluster() returns: the reference's list of 7-tuples in ``estimate_costs`` order
    (cost_het_cluster.py:44-46), as a lazy read-only sequence (the columns live in numpy arrays; strategies /
    partitions stay on the GPU until needed).  ``ranked()`` is ``sorted(result, key=lambda kv: kv[6])``
    (cost_het_cluster.py:76, a stable sort) taken from the device sort's permutation instead of sorting Python
    objects."""

    def __init__(self, candidates, rank_order: Optional[np.ndarray], summary: Dict[str, int],
                 timings: Optional[Dict[str, float]] = None, ranker=None, best_key: Optional[Tuple[int, int]] = None):
        super().__init__(candidates, summary, timings)
        self.rank_order = rank_order          # permutation of sorted(..., key=cost); computed on first use (``ranker``)
        self._ranker = ranker                 # (k=None) -> uint32 permutation (or its first k), from the device
        self._best_key = best_key             # (ordinal, step) of the argmin found by the search kernels

    def ranked(self, k: Optional[int] = None) -> List[Tuple]:
        """The first ``k`` (default: all) entries of ``sorted(result, key=lambda kv: kv[6])``.  Before the whole
        ranking has been asked for, a ``k`` below ``len(self)`` is served by the device selection (only k records
        are ordered)."""
        if self.rank_order is None and self._ranker is not None and k is not None and 0 <= k < len(self):
            return self.candidates.tuples(self._ranker(k))
        if self.rank_order is None:
            self.rank_order = self._ranker() if self._ranker is not None \
                else np.argsort(self.candidates.cost, kind='stable')
            self._ranker = None
        order = self.rank_order
        if k is not None:
            order = order[:k]
        return self.candidates.tuples(order)

    def best(self) -> Optional[Tuple]:
        """argmin (cost, position): the first entry of the ranked list.  The search kernels reduce it on the device
        (het_finalize_kernel: lowest cost, then lowest ordinal, then lowest step), so no sort is needed for it."""
        if self.rank_order is None and self._best_key is not None and len(self):
            rec = self.candidates.records                     # sorted by (ordinal, step): bisect, no temporaries
            want = (int(self._best_key[0]), int(self._best_key[1]))
            lo, hi = 0, len(rec)
            while lo < hi:
                mid = (lo + hi) >> 1
                r = rec[mid]
                if (int(r['ordinal']), int(r['step'])) < want:
                    lo = mid + 1
                else:
                    hi = mid
            if lo < len(rec) and (int(rec[lo]['ordinal']), int(rec[lo]['step'])) == want:
                return self.candidates.tuples([lo])[0]
        top = self.ranked(1)
        return top[0] if top else None


def het_problem(args, gpu_cluster, profile_data, model_config, layer_load_balancer=None,
                node_sequences: Optional[Sequence[Sequence]] = None, corrected: Sequence[str] = (),
                rows_out: Optional[np.ndarray] = None, device_rows: bool = False):
    """Flatten the inputs of cost_het_cluster() (order of ``set(device_types)`` = quirk Q4).  ``device_rows``: the
    host lists only the compositions, the GPU writes the device-group rows (SURVEY.md 8(f)-1)."""
    if node_sequences is None:
        node_sequences = list(permutations(set(gpu_cluster.get_device_types())))
    norm = layer_load_balancer.norm_layer_duration if layer_load_balancer is not None else None
    problem = flatten.build_problem(profile_data, gpu_cluster, model_config, args.gbs,
                                    args.max_profiled_tp_degree, args.max_profiled_batch_size, node_sequences,
                                    norm, corrected=corrected)
    space = flatten.build_plan_space(len(node_sequences), gpu_cluster.get_total_num_devices(), args.gbs,
                                     args.num_layers, args.min_group_scale_variance, args.max_permute_len,
                                     corrected=corrected, rows_out=rows_out, device_rows=device_rows)
    return problem, space, [tuple(s) for s in node_sequences]


# One engine per (device, rank, world): pinned staging arena, device arena, workspace, record / detail buffers.
# cost_het_cluster() is called once per process by the reference's CLI, but a planner service calls it repeatedly;
# the buffers grow to the largest problem seen and are reused (a pinned allocation costs more than a search).
_ENGINES: Dict[Tuple, Tuple] = {}


def _engine(problem, space, device, rank: int, world: int, stride: int):
    from . import search
    dev = search._require_cuda(device)
    key = (dev.index if dev.index is not None else -1, rank, world)
    eng = _ENGINES.get(key)
    if eng is None:
        dp = search.DeviceProblem(problem, space, dev)
        searcher = search.HetSearcher(dp, rank, world, want_records=True, want_detail=True, want_ranking=False,
                                      detail_to_host=False, detail_stride=stride)
        _ENGINES[key] = (dp, searcher)
        return dp, searcher
    dp, searcher = eng
    dp.reload(problem, space)
    if searcher.detail_stride != stride:
        searcher.detail_stride = stride
        searcher.records = searcher.detail = None
    searcher.rebind()
    return dp, searcher


def release_engines() -> None:
    """Drop the cached device / pinned buffers of cost_het_cluster()."""
    _ENGINES.clear()


def _prepare(args, gpu_cluster, profile_data, model_config, layer_load_balancer, node_sequences, device, corrected):
    """What cost_het_cluster() and best_het_plans() share before the search: the corrections are checked, the inputs
    flattened and staged on the device in the cached engine.  Returns (torch.distributed or None, problem, space,
    node sequences, DeviceProblem, HetSearcher, perf_counter() when the flattening ended)."""
    unknown = set(corrected) - {'Q1', 'Q2', 'Q5', 'Q6'}
    if unknown:
        raise ValueError(f'unknown corrections {sorted(unknown)}: choose from Q1, Q2, Q5, Q6')
    import torch
    from . import search
    dist = torch.distributed if (torch.distributed.is_available() and torch.distributed.is_initialized()) else None
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist else (0, 1)
    dev = search._require_cuda(device)
    # the host lists the compositions (a few thousand records); the rows themselves are written by the GPU
    problem, space, seqs = het_problem(args, gpu_cluster, profile_data, model_config, layer_load_balancer,
                                       node_sequences, corrected=tuple(corrected), device_rows=True)
    t1 = time.perf_counter()
    stride = 3 * int(space.blocks['num_stage'].max()) + 1
    dp, searcher = _engine(problem, space, dev, rank, world, stride)
    dp.upload()
    return dist, problem, space, seqs, dp, searcher, t1


def cost_het_cluster(args: argparse.Namespace, gpu_cluster, profile_data: Dict, model_config: ModelConfig,
                     cost_estimator: HeteroCostEstimator, layer_load_balancer: LayerLoadBalancer,
                     node_sequences: Optional[Sequence[Sequence]] = None, device=None,
                     corrected: Sequence[str] = ()) -> HetSearchResult:
    """cost_het_cluster.py:21-50 on the GPU.  Returns the same sequence of
    (node_sequence, device_groups, strategies, batches, layer_partition, num_repartition, cost) in the
    same order (see HetSearchResult).  With torch.distributed initialised the plans are sharded over the ranks and
    every rank returns the full list.

    ``corrected`` (opt-in, default = strict parity with the reference): a subset of ('Q1', 'Q2', 'Q5', 'Q6') - 'Q1'
    drops the mislabelled one-stage block of every node sequence after the first (plan.py:144-148), 'Q2' uses the
    clusterfile's inter_bandwidth between nodes (gpu_cluster.py:56-58 returns the intra value), 'Q5' gives every
    layer to the stage holding most of its seven sub-layers so that none is dropped (load_balancer.py:293-296), 'Q6'
    takes a stage's memory demand from the profile of its own device type (load_balancer.py:41-52 uses the first
    type of the node sequence and, for mixed stages, sums a whole-cluster split).  Results of a corrected search are
    NOT the reference's; ``result.summary['corrected']`` records what was applied."""
    from . import search
    t0 = time.perf_counter()
    dist, problem, space, seqs, dp, searcher, t1 = _prepare(args, gpu_cluster, profile_data, model_config,
                                                            layer_load_balancer, node_sequences, device, corrected)
    failure = None
    out = best = None
    try:
        out = searcher.run()
    except Exception as exc:                                  # noqa: BLE001 - re-raised below on every rank
        if not dist:
            raise
        failure = exc
    if dist:
        # a rank whose search raised must not leave the others waiting in a collective
        summary, best = search.global_exchange(out.summary if out is not None else {}, out.best if out is not None else None,
                                               dp.device, int(failure is not None))
        if summary['any_rank_failed']:
            raise failure if failure is not None else native.MetisNativeError('the search failed on another rank')
        if summary['global_fatal_ordinal'] < 2 ** 62:
            summary.update(fatal_ordinal=summary['global_fatal_ordinal'], fatal_code=summary['global_fatal_code'],
                           fatal_aux=summary['global_fatal_aux'])
        else:
            summary['fatal_ordinal'] = 2 ** 64 - 1
            out = search.gather_records(out, searcher, want_rank=False, counts=summary['records_per_rank'])
    else:
        summary, best = out.summary, out.best
    if summary['fatal_ordinal'] != 2 ** 64 - 1:
        # the reference dies at that plan: nothing is returned (quirk Q8)
        search.raise_fatal(summary, problem)
    t2 = time.perf_counter()
    # the row blob of the engine is rewritten by the next call: a lazy result keeps its own copy (a few MB, on the GPU)
    cand = search.Candidates(out.records, out.detail, space, seqs, detail_dev=out.detail_dev,
                             rows_dev=dp.rows_device().clone())
    # sorted(result, key=cost) is the CALLER's step in the reference (cost_het_cluster.py:76): its permutation is
    # computed by the device sort when ranked() is first asked for; best() needs no sort at all
    result = HetSearchResult(cand, out.rank_order,
                             dict(summary, num_plans=space.num_plans, corrected=tuple(sorted(corrected))),
                             ranker=search.make_ranker(searcher, out.records_dev) if len(out.records) else None,
                             best_key=(best[1], best[2]) if best else None)
    result.timings = {'flatten_enumerate_s': t1 - t0, 'gpu_search_s': t2 - t1,
                      'decode_columns_s': time.perf_counter() - t2}
    return result


# best_het_plans on one GPU: up to this many winners are replayed (metis_het_detail, one thread per winner walks its
# whole strategy chain); more are gathered from detail rows the search writes.  On a B200 the replay of 1000 winners
# cost 16 - 30 ms (profiles/r03_topk.md), more than the whole list's detail rows.
_TOPK_REPLAY_MAX = 64


class HetTopResult(_TupleSequence):
    """What best_het_plans() returns: ``cost_het_cluster(...).ranked(k)`` - the k best 7-tuples in rank order - as a
    lazy read-only sequence.  ``summary`` holds the counters of the WHOLE search (``num_records`` = C, not k)."""


def best_het_plans(args: argparse.Namespace, gpu_cluster, profile_data: Dict, model_config: ModelConfig,
                   cost_estimator: HeteroCostEstimator, layer_load_balancer: LayerLoadBalancer, k: int,
                   node_sequences: Optional[Sequence[Sequence]] = None, device=None,
                   corrected: Sequence[str] = ()) -> HetTopResult:
    """The k best plans of cost_het_cluster() without producing the whole list: equal, tuple for tuple and bit for
    bit, to ``cost_het_cluster(...).ranked(k)`` (lowest cost first, equal costs in estimate_costs order), and
    raising what cost_het_cluster() raises.  The search writes no detail rows, the device selects the k best records
    (metis_select_records), only those k records reach the host and their strategies and partitions are replayed.
    With torch.distributed initialised every rank sends its k best to every other rank (instead of its whole list)
    and every rank returns the same k."""
    k = operator.index(k)
    if k < 0:
        raise ValueError(f'k must be >= 0, got {k}')
    import torch
    from . import search
    t0 = time.perf_counter()
    dist, problem, space, seqs, dp, searcher, t1 = _prepare(args, gpu_cluster, profile_data, model_config,
                                                            layer_load_balancer, node_sequences, device, corrected)
    failure = None
    out = None
    try:
        # one GPU: few winners are replayed, many are gathered from detail rows written during the search
        out = searcher.run_top(k, with_detail=dist is None and k > _TOPK_REPLAY_MAX)
    except Exception as exc:                                  # noqa: BLE001 - re-raised below on every rank
        if not dist:
            raise
        failure = exc
    if dist:
        def select(records, kk):
            return searcher.select_records(records, records.numel() // 2, kk, torch.cuda.current_stream(dp.device))[0]
        summary, _best, top = search.global_top(out.summary if out is not None else {},
                                               out.best if out is not None else None,
                                               out.records_dev if out is not None else None, k, dp.device, failure,
                                               select)
    else:
        summary, top = out.summary, out.records_dev
    if summary['fatal_ordinal'] != 2 ** 64 - 1:
        search.raise_fatal(summary, problem)                  # quirk Q8, as in cost_het_cluster()
    with torch.cuda.device(dp.device):
        records = top.cpu().numpy().view(np.uint8).view(native.RECORD_DTYPE)
        if out is not None and out.detail_dev is not None:
            detail = out.detail_dev.cpu().numpy()
        else:
            detail = searcher.detail_for(records, stride=searcher.detail_stride) if len(records) else None
    t2 = time.perf_counter()
    cand = search.Candidates(records, detail, space, seqs, rows_dev=dp.rows_device().clone())
    return HetTopResult(cand, dict(summary, num_plans=space.num_plans, corrected=tuple(sorted(corrected))),
                        {'flatten_enumerate_s': t1 - t0, 'gpu_search_s': t2 - t1,
                         'decode_columns_s': time.perf_counter() - t2})


def cost_homo_cluster(args: argparse.Namespace, gpu_cluster, cost_estimator: HomoCostEstimator,
                      device_type: Optional[str] = None, device=None) -> List[Tuple[UniformPlan, float]]:
    """cost_homo_cluster.py:21-37 on the GPU: every gbs-matching UniformPlan is costed by
    homo_cost_kernel; plans whose profile key is missing are skipped like ``except KeyError``."""
    from copy import copy
    from . import search
    profile_data = cost_estimator.profile_data
    if device_type is None:
        device_type = next(k for k in profile_data if k.startswith('DeviceType.')).split('.', 1)[1]
    for key in profile_data[f'DeviceType.{device_type}']:
        tp = int(key[2:].split('_bs')[0])
        if tp & (tp - 1):
            raise NotImplementedError(f'profile key {key}: non power-of-two tp is not supported on the GPU path')
    plans = [copy(p) for p in UniformPlanGenerator(num_devices=gpu_cluster.get_total_num_devices(),
                                                   max_tp=args.max_profiled_tp_degree, max_gbs=args.gbs)
             if p.gbs == args.gbs]
    max_tp = max([p.tp for p in plans] + [1])
    max_bs = max([p.mbs for p in plans] + [1])
    cluster_types = [t.name for t in gpu_cluster.get_device_types()]
    problem = flatten.build_problem(profile_data, gpu_cluster, cost_estimator.model_config, args.gbs,
                                    max_tp, max_bs, [tuple(dict.fromkeys(cluster_types))])
    if device_type not in problem.type_names:
        raise KeyError(f'DeviceType.{device_type}')
    table = np.array([[p.dp, p.pp, p.tp, p.mbs, p.gbs] for p in plans], dtype=np.int32).reshape(-1, 5)
    cost, status = search.homo_costs(problem, problem.type_names.index(device_type), table, device)
    return [(p, float(c)) for p, c, s in zip(plans, cost, status) if s != 1]
