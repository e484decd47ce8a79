import hashlib
import json
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, 'golden')
if REPO not in sys.path:
    sys.path.insert(0, REPO)


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box with -m gpu)')
    config.addinivalue_line('markers', 'slow: long-running CPU test')


def load_golden(name):
    """Returns (meta dict, arrays dict) of tests/golden/<name>.npz (made by make_golden.py).

    'groups' (dp * tp of every stage) is rebuilt when the file does not store it.  A golden too large to keep whole
    holds a seeded sample of the candidates, their positions in the whole list in 'rows', and in meta the whole
    list's 'digest' (candidates_digest) and 'best' (cost, ordinal, step)."""
    path = os.path.join(GOLDEN, f'{name}.npz')
    if not os.path.exists(path):
        pytest.skip(f'golden {name}.npz not generated')
    z = np.load(path, allow_pickle=False)
    meta = json.loads(str(z['meta']))
    arrays = {k: z[k] for k in z.files if k != 'meta'}
    if 'groups' not in arrays and 'dp' in arrays:
        arrays['groups'] = arrays['dp'] * arrays['tp']
    return meta, arrays


def candidates_digest(ordinal, step, nrep, nstage, cost, dp, tp, part):
    """sha256 of a whole candidate list in estimate_costs order.  dp / tp are [n, >= S] and part [n, >= S + 1]
    arrays of values (not log2 codes); entries past a row's stage count S are not part of the digest."""
    S = np.asarray(nstage).astype(np.int64)
    h = hashlib.sha256()
    for a in (ordinal, step, nrep, S):
        h.update(np.asarray(a).astype('<i8').tobytes())
    h.update(np.asarray(cost).astype('<f8').tobytes())
    for m, extra in ((dp, 0), (tp, 0), (part, 1)):
        m = np.asarray(m)
        h.update(m[np.arange(m.shape[1])[None, :] < (S + extra)[:, None]].astype('<i8').tobytes())
    return h.hexdigest()


def golden_best(meta, arrays):
    """(cost, ordinal, step) of the golden's best candidate: min by cost, then ordinal, then step."""
    if 'best' in meta:
        return tuple(meta['best'])
    i = int(np.lexsort((arrays['step'], arrays['ordinal'], arrays['cost']))[0])
    return float(arrays['cost'][i]), int(arrays['ordinal'][i]), int(arrays['step'][i])


def device_columns(records, detail, width):
    """Records (native.RECORD_DTYPE) and their detail rows (dp codes[S], tp codes[S], partition[S + 1]) as golden
    columns: dp / tp [n, width] and part [n, width + 1] hold values, zero past each row's stage count."""
    S = records['num_stage'].astype(np.int64)
    rows = np.arange(len(records))[:, None]
    col = np.arange(width + 1)[None, :]
    last = detail.shape[1] - 1

    def take(start, w):
        return detail[rows, np.minimum(start[:, None] + col[:, :w], last)].astype(np.int64)
    live, livep = col[:, :width] < S[:, None], col <= S[:, None]
    return dict(ordinal=records['ordinal'].astype(np.int64), step=records['step'].astype(np.int64),
                nrep=records['num_repartition'].astype(np.int64), nstage=S, cost=records['cost'],
                dp=np.where(live, 1 << take(0 * S, width), 0), tp=np.where(live, 1 << take(S, width), 0),
                part=np.where(livep, take(2 * S, width + 1), 0))


def assert_candidates_equal(got, meta, arrays):
    """``got`` (device_columns of the whole candidate list) equals the golden: every candidate, or, for a sampled
    golden, the candidates at the sampled positions and the digest of the whole list."""
    if 'rows' in arrays:
        assert len(got['cost']) == meta['counters']['C']
        whole = got
        got = {k: v[arrays['rows']] for k, v in got.items()}
    assert len(got['cost']) == len(arrays['cost'])
    assert (got['ordinal'] == arrays['ordinal']).all() and (got['step'] == arrays['step']).all()
    assert (got['nrep'] == arrays['nrep']).all() and (got['nstage'] == arrays['nstage']).all()
    assert (got['cost'].view(np.uint64) == arrays['cost'].view(np.uint64)).all(), 'fp64 cost bits differ'
    width = got['dp'].shape[1]
    assert (got['dp'] == arrays['dp'][:, :width]).all() and (got['tp'] == arrays['tp'][:, :width]).all()
    assert (got['part'] == arrays['part'][:, :width + 1]).all()
    assert (got['dp'] * got['tp'] == arrays['groups'][:, :width]).all()
    if 'rows' in arrays:
        assert candidates_digest(**whole) == meta['digest'], 'candidates outside the stored sample differ'


def golden_rows(arrays):
    """Unpack golden arrays into tuples comparable with oracle / product candidates."""
    out = []
    for i in range(len(arrays['cost'])):
        s = int(arrays['nstage'][i])
        out.append((int(arrays['ordinal'][i]), int(arrays['step'][i]), int(arrays['ns_idx'][i]),
                    [int(x) for x in arrays['groups'][i, :s]],
                    [(int(d), int(t)) for d, t in zip(arrays['dp'][i, :s], arrays['tp'][i, :s])],
                    int(arrays['batches'][i]),
                    [int(x) for x in arrays['part'][i, :s + 1]],
                    int(arrays['nrep'][i]), float(arrays['cost'][i])))
    return out


@pytest.fixture(scope='session')
def workload_dir(tmp_path_factory):
    """Materialise a named synthetic workload once per session; returns (Workload, root)."""
    from metis_b200.workloads import WORKLOADS, materialize
    cache = {}

    def get(name):
        if name not in cache:
            root = str(tmp_path_factory.mktemp(name))
            digest = materialize(WORKLOADS[name], root)
            cache[name] = (WORKLOADS[name], root, digest)
        return cache[name]
    return get


C1_DIR = os.path.join(GOLDEN, 'fixtures', 'c1')
