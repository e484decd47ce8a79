#!/usr/bin/env python3
"""Drop-in CLI for the reference's cost_het_cluster.py (same flags, same stdout);
the search itself runs on the GPU (metis_b200.api.cost_het_cluster).

The reference prints several lines per candidate while it searches (287 MB for 8e4 inter-stage plans).  They are
produced only on request - METIS_VERBOSE=1 - by replaying every plan on the GPU and formatting the recorded values
(metis_b200/verbose.py); with it the whole stdout equals the reference's byte for byte except the search_time line.

METIS_TOP_K=N prints only the first N rows of the ranked table (the rest of stdout is unchanged; `len(costs):` still
counts every candidate) and never builds the whole list: the N best plans are selected on the GPU
(metis_b200.api.best_het_plans)."""
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from metis_b200.api import (GPTActivationAndParam, HeteroCostEstimator, LayerLoadBalancer,  # noqa: E402
                            best_het_plans, cost_het_cluster)
from metis_b200.arguments import parse_args  # noqa: E402
from metis_b200.data_loader import ProfileDataLoader  # noqa: E402
from metis_b200.gpu_cluster import GPUCluster  # noqa: E402
from metis_b200.utils import ModelConfig  # noqa: E402


def top_k_from_env(environ=os.environ):
    """METIS_TOP_K as a row count (None when unset or empty); anything but a non-negative integer is refused."""
    raw = environ.get('METIS_TOP_K', '').strip()
    if not raw:
        return None
    try:
        k = int(raw, 10)
    except ValueError:
        raise ValueError(f'METIS_TOP_K must be a non-negative integer, got {raw!r}') from None
    if k < 0:
        raise ValueError(f'METIS_TOP_K must be a non-negative integer, got {raw!r}')
    return k


def main(argv=None, node_sequences=None, file_order=None):
    """``node_sequences`` / ``file_order`` pin what the reference takes from set() iteration order (quirk Q4) and
    os.listdir order (quirk Q3); by default they are taken like the reference takes them."""
    top_k = top_k_from_env()
    args = parse_args(argv)
    gpu_cluster = GPUCluster(hostfile_path=args.hostfile_path, clusterfile_path=args.clusterfile_path)
    profile_data, _ = ProfileDataLoader(args.profile_data_path, file_order).load_profile_data_all()
    print(profile_data)
    assert len(profile_data.keys()) > 0, 'There is no profiled data at the specified path.'

    model_config = ModelConfig(model_name=args.model_name, num_layers=args.num_layers,
                               sequence_length=args.sequence_length, vocab_size=args.vocab_size,
                               hidden_size=args.hidden_size, attention_head_size=args.attention_head_size)
    model_volume = GPTActivationAndParam(model_config, profile_data['model']['parameters'])
    cost_estimator = HeteroCostEstimator(profile_data, model_config, model_volume, gpu_cluster)
    layer_load_balancer = LayerLoadBalancer(gpu_cluster, profile_data, model_config, args.gbs)

    if os.environ.get('METIS_VERBOSE', '') not in ('', '0'):
        from metis_b200.verbose import plan_transcript
        for line in plan_transcript(args, gpu_cluster, profile_data, model_config, layer_load_balancer, node_sequences):
            print(line)
    start_time = time.time()
    if top_k is None:
        estimate_costs = cost_het_cluster(args, gpu_cluster, profile_data, model_config, cost_estimator,
                                          layer_load_balancer, node_sequences=node_sequences)
    else:
        estimate_costs = best_het_plans(args, gpu_cluster, profile_data, model_config, cost_estimator,
                                        layer_load_balancer, top_k, node_sequences=node_sequences)
    print(f'search_time: {time.time() - start_time}s')
    if top_k is None:
        print(f'len(costs): {len(estimate_costs)}')
        ranked = estimate_costs.ranked()  # = sorted(estimate_costs, key=lambda kv: kv[6]), order from the device sort
    else:
        print(f'len(costs): {estimate_costs.summary["num_records"]}')
        ranked = estimate_costs           # already the first top_k rows of that order
    print('rank, cost, node_sequence, device_groups, strategies(dp_deg, tp_deg), batches(number of batch), '
          'layer_partition')
    for idx, r in enumerate(ranked):
        print(f'{idx + 1}, {r[6]}, {r[0]}, {r[1]}, {r[2]}, {r[3]}, {r[4]}')
    return ranked


if __name__ == '__main__':
    main()
