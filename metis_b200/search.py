"""Device-side plan search: the B200 replacement of the loops in cost_het_cluster.py:21-50
and cost_homo_cluster.py:21-37 of the reference.

PyTorch is used only for device buffers, streams and (multi-GPU) torch.distributed; all
search arithmetic runs in libmetis_b200.so (hand-written sm_100a CUDA) behind the C ABI of
include/metis_b200.h.  There is no CPU path: without CUDA these functions raise.
"""
from __future__ import annotations

import ctypes as C
import weakref
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import flatten, native


def _require_cuda(device) -> torch.device:
    if not torch.cuda.is_available():
        raise native.MetisNativeError('CUDA device required: metis_b200 has no CPU fallback')
    return torch.device(device if device is not None else f'cuda:{torch.cuda.current_device()}')


def _align(n: int, a: int = 256) -> int:
    return (n + a - 1) // a * a


_PROBLEM_ARRAYS = ('key_index', 'layer_compute', 'layer_memory', 'exec_full', 'fb_sync', 'norm_lc', 'type_memory',
                   'type_bw_first', 'type_bw_min', 'ns_run_type', 'ns_run_end', 'ns_q10_end')
# 'rows' is last: spaces whose rows the GPU writes itself (flatten.build_plan_space(device_rows=True)) upload
# everything before it - the composition list instead of the rows - and fill it with metis_generate_rows
_ARENA_ORDER = _PROBLEM_ARRAYS + ('blocks', 'batches', 'comp_recs', 'comp_pool', 'rows')
_EMPTY = np.zeros(0, dtype=np.uint8)


class DeviceProblem:
    """A flattened problem + candidate space resident in HBM (one upload, many searches).

    All tables live in ONE pinned host arena and ONE device arena at the same offsets, so an upload is a single
    host -> device copy; ``reload`` puts another problem / space of compatible size into the same buffers."""

    def __init__(self, problem: flatten.FlatProblem, space: flatten.FlatPlanSpace, device=None,
                 pinned: bool = True, rows_capacity: int = 0):
        self.device = _require_cuda(device)
        self.lib = native.load_library()
        self.pinned = pinned
        self._host = self._dev = None
        self._off: Dict[str, Tuple[int, int]] = {}           # name -> (offset, capacity)
        self._used: Dict[str, int] = {}
        self._allocate(self._arrays(problem, space), space, rows_capacity)
        self.reload(problem, space)
        self.upload()

    @staticmethod
    def _arrays(problem: flatten.FlatProblem, space: flatten.FlatPlanSpace) -> Dict[str, np.ndarray]:
        arrays = {k: problem.arrays[k] for k in _PROBLEM_ARRAYS}
        arrays.update(blocks=space.blocks.view(np.uint8).reshape(-1), batches=space.batches, rows=space.rows,
                      comp_recs=space.comp_recs.view(np.uint8).reshape(-1) if space.comp_recs is not None else _EMPTY,
                      comp_pool=space.comp_pool if space.comp_pool is not None else _EMPTY)
        return {k: np.ascontiguousarray(v).view(np.uint8).reshape(-1) for k, v in arrays.items()}

    @staticmethod
    def _need(flat: Dict[str, np.ndarray], space: flatten.FlatPlanSpace, name: str) -> int:
        if name == 'rows' and space.comp_recs is not None:
            return int(space.rows_total_bytes)               # written by the GPU, never staged on the host
        return int(flat[name].size)

    def _allocate(self, flat: Dict[str, np.ndarray], space: flatten.FlatPlanSpace, rows_capacity: int) -> None:
        off = host_bytes = 0
        self._off = {}
        for name in _ARENA_ORDER:
            need = max(self._need(flat, space, name), 16)
            cap = _align(need + need // 4 if name in ('rows', 'blocks', 'comp_recs', 'comp_pool') else need)
            if name == 'rows':
                cap = max(cap, _align(rows_capacity))
                host_bytes = off + (16 if space.comp_recs is not None and not rows_capacity else cap)
            self._off[name] = (off, cap)
            off += cap
        host = torch.zeros(host_bytes, dtype=torch.uint8)
        self._host = host.pin_memory() if self.pinned else host
        with torch.cuda.device(self.device):
            self._dev = torch.zeros(off, dtype=torch.uint8, device=self.device)

    def fits(self, problem: flatten.FlatProblem, space: flatten.FlatPlanSpace) -> bool:
        flat = self._arrays(problem, space)
        return (all(self._need(flat, space, n) <= self._off[n][1] for n in _ARENA_ORDER)
                and self._off['rows'][0] + flat['rows'].size <= self._host.numel())

    def reload(self, problem: flatten.FlatProblem, space: flatten.FlatPlanSpace) -> None:
        """Stage another problem / space (host side only; call upload()).  Tables that already live in the staging
        arena (``build_plan_space(rows_out=staging('rows'))``) are not copied again."""
        flat = self._arrays(problem, space)
        if not self.fits(problem, space):
            keep = {n: flat[n].copy() for n in _ARENA_ORDER}     # a view into the old arena must survive the swap
            self._allocate(keep, space, 0)
            flat = keep
        host = self._host.numpy()
        for name in _ARENA_ORDER:
            src = flat[name]
            off, _cap = self._off[name]
            dst = host[off:off + src.size]
            if src.size and not np.shares_memory(src, dst):
                dst[:] = src
            self._used[name] = int(src.size)
        self.problem, self.space = problem, space
        base = self._dev.data_ptr()
        self.p_struct = problem.as_struct(lambda n: base + self._off[n][0])
        self.s_struct = space.as_struct(lambda n: base + self._off[n][0])
        self.device_rows = space.comp_recs is not None
        self.h2d_bytes = self._off['rows'][0] + self._used['rows']          # device_rows: nothing of 'rows'

    def staging(self, name: str) -> np.ndarray:
        """The pinned host region of one table (numpy view, full capacity): fill it in place, then upload()."""
        off, cap = self._off[name]
        return self._host.numpy()[off:off + cap]

    def restage_space(self, space: flatten.FlatPlanSpace) -> None:
        """Put a freshly enumerated space into the staging arena (same problem)."""
        self.reload(self.problem, space)

    def upload(self, stream: Optional[torch.cuda.Stream] = None) -> None:
        """Host -> HBM: ONE copy of the arena's used prefix (part of the end-to-end timed region)."""
        n = self.h2d_bytes
        with torch.cuda.device(self.device), torch.cuda.stream(stream or torch.cuda.current_stream(self.device)):
            self._dev[:n].copy_(self._host[:n], non_blocking=True)
            if self.device_rows:                              # SURVEY.md 8(f)-1: the GPU writes the rows itself
                base = self._dev.data_ptr()
                s = torch.cuda.current_stream(self.device)
                rc = self.lib.metis_generate_rows(C.c_void_p(base + self._off['comp_recs'][0]),
                                                  C.c_int64(len(self.space.comp_recs)),
                                                  C.c_void_p(base + self._off['comp_pool'][0]),
                                                  C.c_void_p(base + self._off['rows'][0]), C.c_void_p(s.cuda_stream))
                native.check(rc, 'metis_generate_rows')

    def rows_device(self) -> torch.Tensor:
        """The row blob in HBM (uint8 view; MetisPlanBlock.rows_offset addresses it)."""
        off = self._off['rows'][0]
        n = int(self.space.rows_total_bytes) if self.device_rows else self._used['rows']
        return self._dev[off:off + n]

    def workspace_bytes(self, num_plans: int) -> int:
        n = self.lib.metis_het_workspace_bytes(C.byref(self.p_struct), num_plans, self.s_struct.max_stage)
        if n < 0:
            native.check(int(n), 'metis_het_workspace_bytes')
        return int(n)


@dataclass
class HetSearchOutput:
    """Result of one shard's search.  ``records`` (host, numpy) are in estimate_costs order; ``detail`` rows are
    aligned with them: a numpy array when the searcher copies them to the host, else only ``detail_dev``."""
    summary: Dict[str, int]
    best: Optional[Tuple[float, int, int, int, int]]      # cost, ordinal, step, num_repartition, num_stage
    records: Optional[np.ndarray]                         # native.RECORD_DTYPE sorted by (ordinal, step)
    detail: Optional[np.ndarray]                          # uint8 [n, stride] aligned with records
    d2h_bytes: int = 0
    rank_order: Optional[np.ndarray] = None               # uint32: records[rank_order] = sorted(..., key=cost), stable
    detail_dev: Optional[torch.Tensor] = None             # uint8 [n, stride] on the device
    records_dev: Optional[torch.Tensor] = None            # int64 [2n]: the sorted records on the device


class HetSearcher:
    """Owns the output buffers for repeated searches over one DeviceProblem."""

    def __init__(self, dp: DeviceProblem, rank: int = 0, world: int = 1, tile: int = 128,
                 want_records: bool = True, want_detail: bool = False, capacity: Optional[int] = None,
                 want_ranking: bool = False, detail_to_host: bool = True, detail_stride: Optional[int] = None):
        self.dp = dp
        self.want_ranking = want_ranking and want_records
        self._sort_ws = self._select_ws = None
        self.shard = native.MetisShard(rank, world, tile, 0)
        self.want_records = want_records
        self.want_detail = want_detail and want_records
        self.detail_to_host = detail_to_host
        self.detail_stride = int(detail_stride or native.DETAIL_STRIDE)
        self.capacity = 0
        self.workspace = None
        self.summary_host = torch.zeros(C.sizeof(native.MetisSearchSummary), dtype=torch.uint8).pin_memory()
        self._host_buf: Dict[str, list] = {}                 # name -> [[pinned tensor, weakref to the array handed out]]
        self.records = self.detail = None
        self._fixed_capacity = capacity
        self.rebind()

    def rebind(self) -> None:
        """(Re)size the buffers for the DeviceProblem's current space (after DeviceProblem.reload)."""
        dp = self.dp
        tile, world = self.shard.tile, self.shard.world
        rounds = -(-dp.space.num_plans // (tile * world))
        self.shard_plans = rounds * tile
        need = dp.workspace_bytes(self.shard_plans)
        if self.workspace is None or self.workspace.numel() < need:
            with torch.cuda.device(dp.device):
                self.workspace = torch.empty(need + need // 8, dtype=torch.uint8, device=dp.device)
        if self.want_records and self.records is None:
            self._alloc(self._fixed_capacity if self._fixed_capacity is not None else min(self.shard_plans + 4096, 1 << 18))

    def _alloc(self, capacity: int) -> None:
        dev = self.dp.device
        self.capacity = capacity
        with torch.cuda.device(dev):
            self.records = torch.empty(capacity * 2, dtype=torch.int64, device=dev)
            self.detail = (torch.empty((capacity, self.detail_stride), dtype=torch.uint8, device=dev)
                           if self.want_detail else None)

    def launch(self, stream: Optional[torch.cuda.Stream] = None, with_detail: bool = True) -> None:
        """Enqueue pack + search + finalize + summary copy on ``stream`` (asynchronous)."""
        dp = self.dp
        s = stream or torch.cuda.current_stream(dp.device)
        detail = self.detail if with_detail else None
        rc = dp.lib.metis_het_search(
            C.byref(dp.p_struct), C.byref(dp.s_struct), C.byref(self.shard),
            C.c_void_p(self.records.data_ptr() if self.records is not None else 0), C.c_int64(self.capacity),
            C.c_void_p(detail.data_ptr() if detail is not None else 0), C.c_int32(self.detail_stride),
            C.c_void_p(self.workspace.data_ptr()), C.c_int64(self.workspace.numel()),
            C.c_void_p(self.summary_host.data_ptr()), C.c_void_p(s.cuda_stream))
        native.check(rc, 'metis_het_search')

    def summary(self) -> native.MetisSearchSummary:
        return native.MetisSearchSummary.from_buffer_copy(self.summary_host.numpy().tobytes())

    def _to_host(self, name: str, dev_tensor: torch.Tensor, stream: torch.cuda.Stream) -> np.ndarray:
        """Device -> pinned host memory, handed out WITHOUT another copy.

        A pinned buffer is reused only when the array handed out from it last time is gone (its weak reference is
        dead: numpy views keep their root array alive), so a result a caller still holds is never overwritten; a
        caller that keeps every result makes each call allocate a new buffer (slow, correct)."""
        n = dev_tensor.numel() * dev_tensor.element_size()
        pool = self._host_buf.setdefault(name, [])
        slot = None
        for entry in pool:
            if entry[1] is None or entry[1]() is None:
                if entry[0].numel() >= n:
                    slot = entry
                    break
        if slot is None:
            pool[:] = [e for e in pool if not (e[1] is None or e[1]() is None)]     # too small and free: drop
            slot = [torch.empty(max(n + n // 8, 1 << 16), dtype=torch.uint8).pin_memory(), None]
            pool.append(slot)
        view = slot[0][:n]
        with torch.cuda.stream(stream):
            view.copy_(dev_tensor.reshape(-1).view(torch.uint8), non_blocking=True)
        stream.synchronize()
        arr = view.numpy()
        slot[1] = weakref.ref(arr)
        return arr

    def _search(self, s: torch.cuda.Stream, with_detail: bool = True):
        """launch + synchronise; grows the record buffer and searches again when it was too small."""
        self.launch(s, with_detail)
        s.synchronize()
        sm = self.summary()
        if self.want_records and sm.num_records > self.capacity:
            # C is not known before the first search of a space: size the buffers and search again
            self._alloc(int(sm.num_records) + max(1024, int(sm.num_records) // 64))
            self.launch(s, with_detail)
            s.synchronize()
            sm = self.summary()
        out_summary = dict(num_records=int(sm.num_records), num_partition_calls=int(sm.num_partition_calls),
                           num_balancer_runs=int(sm.num_balancer_runs), num_keyerror=int(sm.num_keyerror),
                           fatal_ordinal=int(sm.fatal_ordinal), fatal_code=int(sm.fatal_code),
                           fatal_aux=int(sm.fatal_aux), num_admitted=int(sm.reserved[0]),
                           num_chained=int(sm.reserved[1]))
        best = None
        if sm.num_records > 0:
            b = sm.best
            best = (float(b.cost), int(b.ordinal), int(b.step), int(b.num_repartition), int(b.num_stage))
        return sm, out_summary, best

    def run_top(self, k: int, stream: Optional[torch.cuda.Stream] = None, with_detail: bool = False) -> HetSearchOutput:
        """The search, then the shard's ``min(k, C)`` first records of the ranked order selected on the device
        (``records_dev``, ranked, still on the device; ``records`` stays None).  Without detail rows the winners'
        strategies and partitions come from ``detail_for`` afterwards; ``with_detail`` (a searcher that has detail
        rows) writes them during the search and gathers the winners' rows into ``detail_dev``."""
        dp = self.dp
        s = stream or torch.cuda.current_stream(dp.device)
        with_detail = with_detail and self.want_detail
        with torch.cuda.device(dp.device):
            _sm, out_summary, best = self._search(s, with_detail=with_detail)
            n = out_summary['num_records']
            top, idx = self.select_records(self.records, n, k, s, want_idx=with_detail)
            detail_dev = self.detail[:n].index_select(0, idx.long()) if with_detail else None
        return HetSearchOutput(out_summary, best, None, None, C.sizeof(native.MetisSearchSummary), records_dev=top,
                               detail_dev=detail_dev)

    def select_records(self, buf: torch.Tensor, n: int, k: int, stream: torch.cuda.Stream, want_idx: bool = False):
        """metis_select_records on the first n records of ``buf`` (asynchronous on ``stream``): the ranked
        ``min(k, n)`` first records as a new int64 tensor, and their positions in ``buf`` (int32 view of the uint32
        indices) when asked."""
        dp = self.dp
        m = min(k, n)
        need = int(dp.lib.metis_select_workspace_bytes(C.c_int64(n), C.c_int64(k)))
        if need < 0:
            native.check(need, 'metis_select_workspace_bytes')
        if self._select_ws is None or self._select_ws.numel() < need:
            self._select_ws = torch.empty(need + need // 8, dtype=torch.uint8, device=dp.device)
        top = torch.empty(2 * max(m, 1), dtype=torch.int64, device=dp.device)
        idx = torch.empty(max(m, 1), dtype=torch.int32, device=dp.device) if want_idx else None
        rc = dp.lib.metis_select_records(C.c_void_p(buf.data_ptr()), C.c_int64(n), C.c_int64(k),
                                         C.c_void_p(top.data_ptr()), C.c_void_p(idx.data_ptr() if idx is not None else 0),
                                         C.c_void_p(self._select_ws.data_ptr()), C.c_int64(self._select_ws.numel()),
                                         C.c_void_p(stream.cuda_stream))
        native.check(rc, 'metis_select_records')
        return top[:2 * m], (idx[:m] if idx is not None else None)

    def run(self, stream: Optional[torch.cuda.Stream] = None) -> HetSearchOutput:
        """launch + synchronise + bring results to the host; grows the record buffer if needed."""
        dp = self.dp
        s = stream or torch.cuda.current_stream(dp.device)
        with torch.cuda.device(dp.device):
            sm, out_summary, best = self._search(s)
            records = detail = rank_order = detail_dev = records_dev = None
            d2h = C.sizeof(native.MetisSearchSummary)
            if self.want_records:
                n = int(sm.num_records)
                # estimate_costs order = (ordinal, step): rank_records_kernel, in place
                order = self.sort_records(n, native.SORT_POSITION, s, want_perm=self.want_detail)
                records_dev = self.records[:2 * n]
                records = self._to_host('records', records_dev, s).view(native.RECORD_DTYPE)
                d2h += n * 16
                if self.want_detail:
                    detail_dev = self.detail[:n].index_select(0, order.long())
                    if self.detail_to_host:
                        detail = self._to_host('detail', detail_dev, s).reshape(n, self.detail_stride)
                        d2h += n * self.detail_stride
                if self.want_ranking:
                    # sorted(estimate_costs, key=cost): stable by cost on a copy of the ordered records
                    by_cost = self.records[:2 * n].clone()
                    perm = self.sort_records(n, native.SORT_BY_COST_STABLE, s, want_perm=True, buf=by_cost)
                    rank_order = self._to_host('rank', perm, s).view(np.uint32)
                    d2h += n * 4
        return HetSearchOutput(out_summary, best, records, detail, d2h, rank_order, detail_dev, records_dev)

    def sort_records(self, n: int, mode: int, stream: torch.cuda.Stream, want_perm: bool = False, buf=None):
        """metis_sort_records on the first n records (device, in place, asynchronous on ``stream``); returns the
        permutation tensor (int32 view of the uint32 indices) when asked."""
        dp = self.dp
        need = int(dp.lib.metis_sort_workspace_bytes(C.c_int64(n)))
        if self._sort_ws is None or self._sort_ws.numel() < need:
            self._sort_ws = torch.empty(need + need // 8, dtype=torch.uint8, device=dp.device)
        perm = torch.empty(max(n, 1), dtype=torch.int32, device=dp.device) if want_perm else None
        buf = self.records if buf is None else buf
        rc = dp.lib.metis_sort_records(C.c_void_p(buf.data_ptr()), C.c_int64(n), C.c_int32(mode),
                                       C.c_void_p(perm.data_ptr() if perm is not None else 0),
                                       C.c_void_p(self._sort_ws.data_ptr()), C.c_int64(self._sort_ws.numel()),
                                       C.c_void_p(stream.cuda_stream))
        native.check(rc, 'metis_sort_records')
        return perm[:n] if perm is not None else None

    def detail_for(self, picks: np.ndarray, stream: Optional[torch.cuda.Stream] = None,
                   stride: int = native.DETAIL_STRIDE) -> np.ndarray:
        """Strategies and partition of chosen records (metis_het_detail replay), ``stride`` bytes per row."""
        dp = self.dp
        s = stream or torch.cuda.current_stream(dp.device)
        n = len(picks)
        with torch.cuda.device(dp.device):
            raw = torch.from_numpy(np.ascontiguousarray(picks).view(np.uint8).reshape(-1).copy()).to(dp.device)
            out = torch.zeros((max(n, 1), stride), dtype=torch.uint8, device=dp.device)
            rc = dp.lib.metis_het_detail(C.byref(dp.p_struct), C.byref(dp.s_struct), C.c_void_p(raw.data_ptr()),
                                         C.c_int64(n), C.c_void_p(out.data_ptr()), C.c_int32(stride),
                                         C.c_void_p(self.workspace.data_ptr()), C.c_int64(self.workspace.numel()),
                                         C.c_void_p(s.cuda_stream))
            native.check(rc, 'metis_het_detail')
            s.synchronize()
            return out[:n].cpu().numpy()


def raise_fatal(summary: Dict[str, int], problem: flatten.FlatProblem) -> None:
    """Re-raise what the reference would have raised at the first failing plan (quirk Q8)."""
    code = summary['fatal_code']
    if summary['fatal_ordinal'] == 2 ** 64 - 1 or code == 0:
        return
    aux = summary['fatal_aux']
    tp, bs = 1 << ((aux >> 16) & 0xFF), aux & 0xFFFF
    if code in (1, 2):
        raise KeyError(f'tp{tp}_bs{bs}')
    if code == 3:
        raise IndexError('list index out of range')
    if code == 6:
        raise ZeroDivisionError('float division by zero')
    raise RuntimeError(f'plan {summary["fatal_ordinal"]}: {native.FATAL_NAMES.get(code, code)} '
                       f'(the reference does not complete this search either)')


class Candidates:
    """Vectorised view of the costed candidates: every column of the reference's 7-tuples
    (cost_het_cluster.py:44-46) as a numpy array, the tuples themselves built on demand.

    ``detail`` rows hold dp codes[S], tp codes[S] (log2) and layer_partition[S+1]; they may still be on the device
    (``detail_dev``): rows are then fetched per request (a ranked slice costs one small gather + copy), or all at
    once the first time more than a few thousand are needed."""

    _BULK = 4096

    def __init__(self, records: np.ndarray, detail: Optional[np.ndarray], space: flatten.FlatPlanSpace,
                 node_sequences: Sequence[Tuple], detail_dev: Optional[torch.Tensor] = None,
                 rows_dev: Optional[torch.Tensor] = None):
        self.records = records
        self.space = space
        self.node_sequences = [tuple(s) for s in node_sequences]
        self._detail = detail
        self._detail_dev = detail_dev
        # device-group rows: the blob the GPU wrote (``rows_dev``, SURVEY.md 8(f)-1) or the host enumerator's
        self._rows_dev = rows_dev
        self._rows = None if rows_dev is not None else space.host_rows()
        self.cost = records['cost']

    def columns(self, idx=None) -> Dict[str, np.ndarray]:
        """ns_idx, num_stage, row (dg_idx), batches, num_repartition of the candidates ``idx`` (default: all)."""
        rec = self.records if idx is None else self.records[idx]
        blocks = self.space.blocks
        ordinal = rec['ordinal'].astype(np.int64)
        blk = (np.searchsorted(blocks['first_ordinal'], ordinal, side='right') - 1) if len(rec) \
            else np.zeros(0, dtype=np.int64)
        rel = ordinal - blocks['first_ordinal'][blk]
        ndiv = len(self.space.batches)
        row, stages = rel // ndiv, blocks['num_stage'][blk].astype(np.int64)
        return dict(row=row, batches=self.space.batches[rel % ndiv].astype(np.int64),
                    ns_idx=blocks['ns_idx'][blk].astype(np.int64), num_stage=stages,
                    row_byte=blocks['rows_offset'][blk].astype(np.int64) + row * stages,
                    num_repartition=rec['num_repartition'].astype(np.int64))

    def group_codes(self, row_byte: np.ndarray, stages: np.ndarray) -> np.ndarray:
        """log2(device count) of every stage, uint8 [n, max stages] (columns past a row's stage count are junk)."""
        width = int(stages.max())
        at = row_byte[:, None] + np.arange(width, dtype=np.int64)[None, :]
        if self._rows is None:
            if len(row_byte) > self._BULK:
                self._rows = self._rows_dev.cpu().numpy()
                self._rows_dev = None
            else:
                sel = torch.from_numpy(np.minimum(at, self._rows_dev.numel() - 1)).to(self._rows_dev.device)
                return self._rows_dev[sel].cpu().numpy()
        return self._rows[np.minimum(at, len(self._rows) - 1)]

    def __len__(self) -> int:
        return len(self.records)

    def detail_rows(self, idx: np.ndarray) -> np.ndarray:
        if self._detail is None:
            if self._detail_dev is None:
                raise ValueError('the search was run without detail rows')
            if len(idx) > self._BULK:
                self._detail = self._detail_dev.cpu().numpy()
                self._detail_dev = None
            else:
                sel = torch.from_numpy(np.ascontiguousarray(idx, dtype=np.int64)).to(self._detail_dev.device)
                return self._detail_dev.index_select(0, sel).cpu().numpy()
        return self._detail[idx]

    def tuples(self, idx) -> List[Tuple]:
        """The reference's 7-tuples of the candidates ``idx`` (any integer sequence)."""
        idx = np.asarray(idx, dtype=np.int64).reshape(-1)
        if not len(idx):
            return []
        det = self.detail_rows(idx)
        col = self.columns(idx)
        cost = self.cost[idx]
        out = []
        codes = self.group_codes(col['row_byte'], col['num_stage'])
        for k in range(len(idx)):
            S = int(col['num_stage'][k])
            d = det[k]
            groups = (1 << codes[k, :S].astype(np.int64)).tolist()
            dp = (1 << d[:S].astype(np.int64)).tolist()
            tp = (1 << d[S:2 * S].astype(np.int64)).tolist()
            part = d[2 * S:3 * S + 1].astype(np.int64).tolist()
            out.append((self.node_sequences[int(col['ns_idx'][k])], groups, list(zip(dp, tp)), int(col['batches'][k]),
                        part, int(col['num_repartition'][k]), float(cost[k])))
        return out


def materialize(records: np.ndarray, detail: np.ndarray, space: flatten.FlatPlanSpace,
                node_sequences: Sequence[Tuple]) -> List[Tuple]:
    """Records -> the reference's 7-tuples (cost_het_cluster.py:44-46), all of them, eagerly."""
    cand = Candidates(records, detail, space, node_sequences)
    return cand.tuples(np.arange(len(records)))


# ---------------------------------------------------------------------------------------------
# multi-GPU: shard by plan ordinal, one collective at the end (SURVEY.md section 8e)
# ---------------------------------------------------------------------------------------------
def _gather_rows(vec: torch.Tensor) -> torch.Tensor:
    """all_gather of one small vector per rank -> [world, len] on the host (ONE collective, one synchronisation)."""
    import torch.distributed as dist
    world = dist.get_world_size()
    out = torch.empty(world * vec.numel(), dtype=vec.dtype, device=vec.device)
    dist.all_gather_into_tensor(out, vec)
    return out.view(world, vec.numel()).cpu()


_NO_ORDINAL = 2 ** 40
_COUNTER_KEYS = ['num_records', 'num_partition_calls', 'num_balancer_runs', 'num_keyerror']


def _best_row(local_best: Optional[Tuple[float, int, int, int, int]]) -> List[int]:
    """(cost bits, ordinal, step, meta) as int64; a rank without records sends an ordinal nobody has."""
    if local_best is None:
        return [0, _NO_ORDINAL, 0, 0]
    cost, ordinal, step, nrep, nstage = local_best
    return [int(np.array([cost], dtype=np.float64).view(np.int64)[0]), int(ordinal), int(step), int(nrep) * 256 + int(nstage)]


def _pick_best(rows: List[List[int]]) -> Optional[Tuple]:
    """Exact lexicographic min of (cost, ordinal, step) over the ranks' bests."""
    cand = []
    for bits, o, st, m in rows:
        if o < _NO_ORDINAL:
            cand.append((float(np.array([bits], dtype=np.int64).view(np.float64)[0]), int(o), int(st), int(m)))
    if not cand:
        return None
    c, o, st, m = min(cand, key=lambda r: (r[0], r[1], r[2]))
    return (c, o, st, m // 256, m % 256)


def _merge_counters(summary: Dict[str, int], rows: List[List[int]]) -> Dict[str, int]:
    """rows[r] = counters (4), error flag, fatal ordinal, fatal code, fatal aux of rank r."""
    out = dict(summary)
    for i, k in enumerate(_COUNTER_KEYS):
        out[k] = int(sum(r[i] for r in rows))
    out['records_per_rank'] = [int(r[0]) for r in rows]
    out['any_rank_failed'] = int(sum(r[4] for r in rows))
    fatal = [(r[5], r[6], r[7]) for r in rows if r[5] < _NO_ORDINAL]
    if fatal:
        fo, code, aux = min(fatal)                            # the lowest ordinal, with ITS code and aux
        out.update(global_fatal_ordinal=int(fo), global_fatal_code=int(code), global_fatal_aux=int(aux))
    else:
        out.update(global_fatal_ordinal=2 ** 62, global_fatal_code=0, global_fatal_aux=0)
    return out


def _counter_row(summary: Dict[str, int], local_error: int) -> List[int]:
    fo = min(summary.get('fatal_ordinal', 2 ** 64 - 1), _NO_ORDINAL)
    return [int(summary.get(k, 0)) for k in _COUNTER_KEYS] + \
        [int(local_error != 0), int(fo), int(summary.get('fatal_code', 0)) & 0xFF, int(summary.get('fatal_aux', 0))]


def global_best(local_best: Optional[Tuple[float, int, int, int, int]], device) -> Optional[Tuple]:
    """all_gather of one (cost, ordinal, step, meta) record per rank, then the exact lexicographic min."""
    rows = _gather_rows(torch.tensor(_best_row(local_best), dtype=torch.int64, device=device)).tolist()
    return _pick_best(rows)


def global_counters(summary: Dict[str, int], device, local_error: int = 0) -> Dict[str, int]:
    """Sum of the counters over the ranks, the records of every rank, the lowest fatal ordinal with ITS code and aux,
    and an error flag (``any_rank_failed``) so that a rank whose search raised makes every rank raise instead of
    leaving the others in a collective."""
    rows = _gather_rows(torch.tensor(_counter_row(summary, local_error), dtype=torch.int64, device=device)).tolist()
    return _merge_counters(summary, rows)


def global_exchange(summary: Dict[str, int], local_best, device, local_error: int = 0):
    """global_counters and global_best in ONE collective (the API path)."""
    vec = torch.tensor(_counter_row(summary, local_error) + _best_row(local_best), dtype=torch.int64, device=device)
    rows = _gather_rows(vec).tolist()
    return _merge_counters(summary, [r[:8] for r in rows]), _pick_best([r[8:] for r in rows])


def global_top(summary: Dict[str, int], local_best, local_top: Optional[torch.Tensor], k: int, device,
               failure: Optional[BaseException] = None, select=None):
    """The multi-rank step of a top-k search.  The counters, the error flag and the fatal plan travel in the one
    96-byte ``global_exchange``; a rank whose search raised (``failure``) makes every rank raise.  Without a fatal
    plan each rank's ``min(k, C_r)`` ranked records (``local_top``: int64 [2 m] on ``device``) are all-gathered,
    k slots per rank, and ``select(records, k)`` picks the global first k from the merged ones.  Returns
    (summary, best, top records or None when a plan was fatal)."""
    import torch.distributed as dist
    merged, best = global_exchange(summary, local_best, device, int(failure is not None))
    if merged['any_rank_failed']:
        raise failure if failure is not None else native.MetisNativeError('the search failed on another rank')
    if merged['global_fatal_ordinal'] < 2 ** 62:
        merged.update(fatal_ordinal=merged['global_fatal_ordinal'], fatal_code=merged['global_fatal_code'],
                      fatal_aux=merged['global_fatal_aux'])
        return merged, best, None
    merged['fatal_ordinal'] = 2 ** 64 - 1
    world = dist.get_world_size()
    counts = [min(k, c) for c in merged['records_per_rank']]
    cap = max(max(counts), 1)
    mine = counts[dist.get_rank()]
    pad = torch.zeros(2 * cap, dtype=torch.int64, device=device)
    pad[:2 * mine] = local_top[:2 * mine]
    gathered = torch.empty(2 * cap * world, dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(gathered, pad)
    every = torch.cat([gathered[2 * cap * r:2 * cap * r + 2 * counts[r]] for r in range(world)]).contiguous()
    return merged, best, select(every, k)


def make_ranker(searcher: 'HetSearcher', records_dev: torch.Tensor):
    """(k=None) -> permutation of ``sorted(records, key=cost)`` (stable), or its first k entries: the device sort, or
    for a k the device selection, on a private copy of the ordered records, run when a caller first asks."""
    snap = records_dev.clone()
    n = snap.numel() // 2
    dev = searcher.dp.device

    def rank(k: Optional[int] = None) -> np.ndarray:
        with torch.cuda.device(dev):
            s = torch.cuda.current_stream(dev)
            if k is None:
                perm = searcher.sort_records(n, native.SORT_BY_COST_STABLE, s, want_perm=True, buf=snap)
            else:
                # the records are in position order, so the selection's input positions index estimate_costs
                _, perm = searcher.select_records(snap, n, k, s, want_idx=True)
            s.synchronize()
            return perm.cpu().numpy().view(np.uint32)
    return rank


def gather_records(out: HetSearchOutput, searcher: HetSearcher, want_rank: bool = True,
                   counts: Optional[List[int]] = None) -> HetSearchOutput:
    """Every rank receives every rank's records (+ detail rows): padded tensor all_gathers over NCCL (no pickling),
    then the merged list is put into estimate_costs order and ranked by the device sort."""
    import torch.distributed as dist
    dev = searcher.dp.device
    world = dist.get_world_size()
    n_local = len(out.records)
    if counts is None:                                        # records of every rank (global_counters has them too)
        mine = torch.zeros(world, dtype=torch.int64, device=dev)
        mine[dist.get_rank()] = n_local
        dist.all_reduce(mine, op=dist.ReduceOp.SUM)
        counts = mine.cpu().tolist()
    cap = max(max(counts), 1)
    stride = searcher.detail_stride
    with torch.cuda.device(dev):
        rec_pad = torch.empty(cap * 2, dtype=torch.int64, device=dev)
        rec_pad[:2 * n_local] = out.records_dev
        rec_g = torch.empty(world * cap * 2, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(rec_g, rec_pad)
        rec_all = torch.cat([rec_g[2 * cap * r:2 * cap * r + 2 * counts[r]] for r in range(world)]).contiguous()
        det_all = None
        if out.detail_dev is not None:
            det_pad = torch.empty((cap, stride), dtype=torch.uint8, device=dev)
            det_pad[:n_local] = out.detail_dev
            det_g = torch.empty((world * cap, stride), dtype=torch.uint8, device=dev)
            dist.all_gather_into_tensor(det_g, det_pad)
            det_all = torch.cat([det_g[cap * r:cap * r + counts[r]] for r in range(world)])
        n = sum(counts)
        s = torch.cuda.current_stream(dev)
        perm = searcher.sort_records(n, native.SORT_POSITION, s, want_perm=True, buf=rec_all)
        records = searcher._to_host('records_all', rec_all[:2 * n], s).view(native.RECORD_DTYPE)
        detail_dev = det_all.index_select(0, perm.long()) if det_all is not None else None
        rank_order = None
        if want_rank:
            by_cost = rec_all[:2 * n].clone()
            rank = searcher.sort_records(n, native.SORT_BY_COST_STABLE, s, want_perm=True, buf=by_cost)
            rank_order = searcher._to_host('rank_all', rank, s).view(np.uint32)
        detail = None
        if detail_dev is not None and searcher.detail_to_host:
            detail = searcher._to_host('detail_all', detail_dev, s).reshape(n, stride)
    return HetSearchOutput(out.summary, out.best, records, detail, out.d2h_bytes, rank_order, detail_dev,
                           rec_all[:2 * n])


# ---------------------------------------------------------------------------------------------
# homogeneous path
# ---------------------------------------------------------------------------------------------
def homo_costs(problem: flatten.FlatProblem, type_id: int, plans: np.ndarray, device=None
               ) -> Tuple[np.ndarray, np.ndarray]:
    """HomoCostEstimator.get_cost for every row (dp, pp, tp, mbs, gbs) of ``plans`` on the GPU."""
    dev = _require_cuda(device)
    lib = native.load_library()
    with torch.cuda.device(dev):
        tens = {k: torch.from_numpy(np.ascontiguousarray(v).view(np.uint8).reshape(-1).copy()).to(dev)
                for k, v in problem.arrays.items()}
        p = problem.as_struct(lambda n: tens[n].data_ptr())
        ws = torch.empty(int(lib.metis_het_workspace_bytes(C.byref(p), 0, 1)), dtype=torch.uint8, device=dev)
        n = len(plans)
        d_plans = torch.from_numpy(np.ascontiguousarray(plans, dtype=np.int32).reshape(-1)).to(dev)
        cost = torch.zeros(max(n, 1), dtype=torch.float64, device=dev)
        status = torch.zeros(max(n, 1), dtype=torch.int32, device=dev)
        s = torch.cuda.current_stream(dev)
        rc = lib.metis_homo_cost(C.byref(p), C.c_int32(type_id), C.c_void_p(d_plans.data_ptr()), C.c_int64(n),
                                 C.c_void_p(cost.data_ptr()), C.c_void_p(status.data_ptr()),
                                 C.c_void_p(ws.data_ptr()), C.c_int64(ws.numel()), C.c_void_p(s.cuda_stream))
        native.check(rc, 'metis_homo_cost')
        s.synchronize()
        return cost[:n].cpu().numpy(), status[:n].cpu().numpy()


def layer_balance(capa_rows: Sequence[Sequence[float]], lc: Sequence[float], num_layers: int, device=None
                  ) -> List[List[int]]:
    """LayerComputeBalancer.run for many capacity vectors on the GPU (unit-level entry point)."""
    dev = _require_cuda(device)
    lib = native.load_library()
    n = len(capa_rows)
    stride = max(len(c) for c in capa_rows)
    capa = np.zeros((n, stride))
    ns = np.zeros(n, dtype=np.int32)
    for i, c in enumerate(capa_rows):
        capa[i, :len(c)] = c
        ns[i] = len(c)
    with torch.cuda.device(dev):
        d_capa = torch.from_numpy(capa).to(dev)
        d_ns = torch.from_numpy(ns).to(dev)
        d_lc = torch.tensor(list(lc), dtype=torch.float64, device=dev)
        out = torch.zeros((n, stride + 1), dtype=torch.int16, device=dev)
        ws = torch.empty(len(lc) * 8 + 512, dtype=torch.uint8, device=dev)
        s = torch.cuda.current_stream(dev)
        rc = lib.metis_layer_balance(C.c_void_p(d_capa.data_ptr()), C.c_void_p(d_ns.data_ptr()), C.c_int64(n),
                                     C.c_int32(stride), C.c_void_p(d_lc.data_ptr()), C.c_int32(len(lc)),
                                     C.c_int32(num_layers), C.c_void_p(out.data_ptr()), C.c_void_p(ws.data_ptr()),
                                     C.c_int64(ws.numel()), C.c_void_p(s.cuda_stream))
        native.check(rc, 'metis_layer_balance')
        s.synchronize()
        res = out.cpu().numpy().view(np.uint16)
    return [res[i, :ns[i] + 1].tolist() for i in range(n)]
