"""Unit-level golden vectors (tests/golden/units.json.gz, made by make_golden.py from the reference).

The file stores the reference's outputs only.  The inputs of the LayerComputeBalancer.run and
_adj_compute_performance cases are drawn from random.Random(7) by the functions below, which make_golden.py
uses too; IEEE arithmetic and the Mersenne twister make them the same bits on every machine.
"""
import gzip
import json
import os
import random

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'units.json.gz')


def balancer_inputs(rng):
    """3000 (S, L, capa, lc) cases of LayerComputeBalancer.run."""
    out = []
    for _ in range(3000):
        L = rng.choice([6, 10, 12, 24, 33, 48, 80, 96])
        S = rng.randint(1, min(L, 40))
        lc = [0.02 + rng.random() * 0.05] + [1 + rng.random() * rng.choice([0.01, 0.3, 3.0]) for _ in range(L - 2)] + [0.03]
        tot = sum(lc)
        lc = [x / tot for x in lc]
        mode = rng.random()
        if mode < 0.4:
            capa = [rng.random() + 0.05 for _ in range(S)]
        elif mode < 0.7:
            capa = [rng.choice([1.0, 2.0, 4.0]) for _ in range(S)]
        else:
            capa = [1.0 + 0.02 * rng.random() for _ in range(S)]
        tc = sum(capa)
        capa = [c / tc for c in capa]
        if rng.random() < 0.15:
            capa = [c * rng.uniform(0.5, 1.5) for c in capa]       # un-normalised (after re-weighting)
        out.append((S, L, capa, lc))
    return out


def adjust_inputs(rng):
    """1500 (c, mc, md) cases of LayerLoadBalancer._adj_compute_performance."""
    out = []
    for _ in range(1500):
        S = rng.randint(1, 24)
        c = [rng.random() + 0.01 for _ in range(S)]
        t = sum(c)
        c = [x / t for x in c]
        mc = [rng.choice([16384, 81920, 163840, 655360]) for _ in range(S)]
        md = [0.001 + 5.0 * rng.random() * rng.choice([2e4, 1e5, 4e5]) for _ in range(S)]
        out.append((c, mc, md))
    return out


def unit_inputs():
    """(balancer cases, adjust cases), drawn in this order from one random.Random(7)."""
    rng = random.Random(7)
    bal = balancer_inputs(rng)
    return bal, adjust_inputs(rng)


def load_units():
    """The cases in the form the tests read: device_groups as stored; balancer and adjust with their seeded inputs
    (floats as hex strings) next to the reference's outputs."""
    with gzip.open(PATH, 'rt') as fh:
        stored = json.load(fh)
    bal, adj = unit_inputs()
    assert len(bal) == len(stored['balancer_part']) and len(adj) == len(stored['adjust_out'])
    return {
        'device_groups': stored['device_groups'],
        'balancer': [{'L': L, 'S': S, 'lc': [x.hex() for x in lc], 'capa': [c.hex() for c in capa], 'part': part}
                     for (S, L, capa, lc), part in zip(bal, stored['balancer_part'])],
        'adjust': [{'c': [x.hex() for x in c], 'mc': mc, 'md': [x.hex() for x in md], 'out': out}
                   for (c, mc, md), out in zip(adj, stored['adjust_out'])],
    }
