/*
 * metis_b200.h - C ABI of libmetis_b200.so (hand-written sm_100a CUDA).
 *
 * The reference (SamsungLabs/Metis @ ed41176) is pure Python and has no FFI
 * layer; its seam for the plan-search hot path is the pair of Python functions
 *     cost_het_cluster(args, gpu_cluster, profile_data, model_config,
 *                      cost_estimator, layer_load_balancer)   cost_het_cluster.py:21-50
 *     cost_homo_cluster(args, gpu_cluster, cost_estimator)    cost_homo_cluster.py:21-37
 * Each entry point below replaces the body of one of those loops (or one of the
 * functions they call); INTEGRATION.md shows the ctypes stub a maintainer would
 * add to the reference.  Conventions:
 *   - plain pointers and sizes only; every buffer is caller-allocated and
 *     caller-freed; pointers marked [device] must be CUDA device memory on the
 *     current device, [host] ordinary (ideally pinned) host memory;
 *   - every call only ENQUEUES work on `stream` (a cudaStream_t passed as
 *     void*, NULL = default stream) and returns; results are valid after the
 *     caller synchronises that stream;
 *   - return value 0 on success, a negative METIS_E_* code otherwise; the
 *     library never throws and keeps no global state;
 *   - no CPU fallback exists: without a CUDA device every compute entry point
 *     returns METIS_E_CUDA.
 */
#ifndef METIS_B200_H
#define METIS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define METIS_ABI_VERSION 2

/* return codes */
#define METIS_OK            0
#define METIS_E_CUDA       -1   /* CUDA runtime error (see metis_last_error) */
#define METIS_E_ARG        -2   /* bad argument / unsupported size            */
#define METIS_E_CAPACITY   -3   /* caller buffer too small                    */

/* per-plan fatal codes (the reference would abort the whole search, quirk Q8) */
#define METIS_FATAL_NONE        0
#define METIS_FATAL_KEY_EXEC    1   /* KeyError 'tp{t}_bs{b}' in StagePerformance (model/device_group.py:38,49,79) */
#define METIS_FATAL_KEY_MEMORY  2   /* KeyError in _get_stage_memory_demand (model/load_balancer.py:43,51)          */
#define METIS_FATAL_INDEX       3   /* IndexError: fewer profiled layers than --num_layers (load_balancer.py:219)   */
#define METIS_FATAL_HANG        4   /* reference loop at load_balancer.py:96-104 would not terminate                */
#define METIS_FATAL_SCRATCH     5   /* internal scratch exceeded (more stages / leftovers than compiled limits)     */
#define METIS_FATAL_ZERODIV     6   /* ZeroDivisionError in the reference (zero profiled time / zero total)         */

/* MetisProblem.corrected bits (SURVEY.md 8(f)-4; never set by default) */
#define METIS_FIX_Q5  1   /* a layer goes to the stage holding MOST of its 7 sub-layers (lowest stage on ties):
                             no layer is dropped (the reference keeps only count > 3.5, load_balancer.py:293-296) */
#define METIS_FIX_Q6  2   /* memory demand from the profile of the stage's OWN device type; mixed-type stage:
                             largest replica instead of the sum over a whole-cluster split (load_balancer.py:41-52) */

/* limits compiled into the kernels */
#define METIS_MAX_TYPES   8
#define METIS_MAX_STAGES  128
#define METIS_MAX_LAYERS  256   /* scratch size; --num_layers itself is limited to 255 (one-byte partition entries) */

/*
 * Flattened search problem: the dict-of-dicts `profile_data` (data_loader.py:39-61),
 * `GPUCluster` (gpu_cluster.py:8-58), `ModelConfig` / `GPTActivationAndParam`
 * (utils.py:72-79, model/activation_parameter.py:5-51) and the flags read on the
 * hot path (cost_het_cluster.py:25-36) as dense arrays.
 *
 * A profile key 'tp{t}_bs{b}' of device type d is  key_index[(d*num_tp + log2(t))*num_bs + (b-1)]
 * (-1 = not profiled).  Layer tables are zero-padded to `lpad` entries.
 */
typedef struct MetisProblem {
    int32_t num_types;            /* distinct device types in the cluster                          */
    int32_t num_tp;               /* tp levels 1,2,4,.. covered by key_index                        */
    int32_t num_bs;               /* batch sizes 1..num_bs covered by key_index                     */
    int32_t num_keys;             /* profiled (type,tp,bs) keys                                     */
    int32_t lpad;                 /* padded length of the per-layer tables                          */
    int32_t num_layers;           /* --num_layers                                                   */
    int32_t norm_len;             /* len(norm_layer_duration)  (load_balancer.py:22-27)             */
    int32_t gbs;                  /* --gbs                                                          */
    int32_t max_tp;               /* --max_profiled_tp_degree                                       */
    int32_t max_bs;               /* --max_profiled_batch_size                                      */
    int32_t num_nodes;            /* gpu_cluster.get_num_nodes()                                    */
    int32_t devices_per_node;     /* gpu_cluster.get_num_devices_per_node() (node 0, quirk Q10)     */
    int32_t total_devices;
    int32_t num_node_sequences;
    int32_t uniform_bw;           /* 1 when every type has the same first/min bandwidth             */
    int32_t q10_devices;          /* num_nodes x devices of node 0: length of the rank lists the reference builds
                                     with node 0's GPU count (load_balancer.py:109-119, cluster_bandwidth.py:34-47;
                                     quirk Q10); == total_devices when every node has the same count   */
    int32_t corrected;            /* opt-in deviations from the reference (0 = strict parity): METIS_FIX_* bits  */
    int32_t reserved1;
    int64_t sequence_length, hidden_size, vocab_size;
    double optimizer_time;        /* profile_data['model']['optimizer_time'] (= 2 x optimizer_time_ms) */
    double batch_generator;       /* profile_data['model']['batch_generator']                       */
    double input_params, transformer_params, output_params;   /* activation_parameter.py:22-24      */
    double node0_bandwidth;       /* gpu_cluster.get_intra_bandwidth(0) (homo path, cluster_bandwidth.py:75-76) */
    double node0_memory;          /* gpu_cluster.get_device_memory(0)   (cost_estimator.py:31-32)    */
    const int16_t *key_index;     /* [device] [num_types][num_tp][num_bs]                           */
    const double *layer_compute;  /* [device] [num_keys][lpad]  'layer-computes'                    */
    const double *layer_memory;   /* [device] [num_keys][lpad]  'memory'                            */
    const double *exec_full;      /* [device] [num_keys]  sum(layer-computes)   (Python sum, host)  */
    const double *fb_sync;        /* [device] [num_keys]  0.0 = falsy -> KeyError (quirk Q9)        */
    const double *norm_lc;        /* [device] [norm_len]                                            */
    const double *type_memory;    /* [device] [num_types] get_device_memory_for_device_type()       */
    const double *type_bw_first;  /* [device] [num_types] _get_intra_bandwidth(type)                */
    const double *type_bw_min;    /* [device] [num_types] _get_inter_bandwidth([type]) (quirk Q2)   */
    const uint8_t *ns_run_type;   /* [device] [num_node_sequences][num_types] type id of k-th run   */
    const int32_t *ns_run_end;    /* [device] [num_node_sequences][num_types] cumulative rank count */
    const int32_t *ns_q10_end;    /* [device] [num_node_sequences][num_types] cumulative (nodes of the type x devices of
                                     node 0): the type runs of the Q10 rank list                        */
} MetisProblem;

/* One block of inter-stage plans sharing (ns_idx, num_stage): plan.py:153-175 incl. quirk Q1. */
typedef struct MetisPlanBlock {
    int64_t first_ordinal;        /* ordinal of (row 0, batches = gbs)                              */
    int64_t rows_offset;          /* byte offset of row 0 in MetisPlanSpace.rows                    */
    int32_t num_rows;             /* device-group rows in the block                                 */
    int16_t ns_idx;
    int16_t label_stage;          /* InterStagePlan.num_stage as emitted (1 for Q1 blocks)          */
    int16_t num_stage;            /* len(device_groups)                                             */
    int16_t reserved[3];
} MetisPlanBlock;

/*
 * The enumerated candidate space.  ordinal = first_ordinal + row*num_div + div_idx
 * reproduces the order of InterStagePlanGenerator.__next__ (plan.py:153-175).
 * Rows hold log2(group size), one byte per stage (device_group.py:93-107 order).
 */
typedef struct MetisPlanSpace {
    int64_t num_plans;
    int64_t rows_bytes;           /* size of the `rows` blob (must stay below 4 GiB)                   */
    int32_t num_blocks;
    int32_t num_div;
    int32_t max_stage;            /* largest num_stage of any block (sizes the per-plan task state)  */
    int32_t reserved;
    const MetisPlanBlock *blocks; /* [device] [num_blocks]                                          */
    const int32_t *batches;       /* [device] [num_div] divisors of gbs, descending (plan.py:120-124) */
    const uint8_t *rows;          /* [device]                                                       */
} MetisPlanSpace;

/* 16-byte record per costed candidate (one per estimate_costs.append, cost_het_cluster.py:44-46). */
typedef struct MetisRecord {
    double cost;
    uint32_t ordinal;             /* inter-stage plan ordinal                                       */
    uint16_t step;                /* index of the yield inside the plan's intra-stage chain         */
    uint8_t num_repartition;      /* IntraStagePlan.num_repartition (1..3)                          */
    uint8_t num_stage;
} MetisRecord;

/* Summary written to host memory by metis_het_search (valid after stream sync). */
typedef struct MetisSearchSummary {
    uint64_t num_records;         /* C: candidates costed (may exceed record capacity: then truncated) */
    uint64_t num_partition_calls; /* B: LayerLoadBalancer.partition_layer invocations               */
    uint64_t num_balancer_runs;   /* LayerComputeBalancer.run invocations                           */
    uint64_t num_keyerror;        /* candidates skipped by `except KeyError` (cost_het_cluster.py:47) */
    uint64_t fatal_ordinal;       /* lowest ordinal that hit a fatal condition, UINT64_MAX if none  */
    uint32_t fatal_code;          /* METIS_FATAL_* of that ordinal                                  */
    uint32_t fatal_aux;           /* tp<<16 | bs of the missing key when applicable                 */
    MetisRecord best;             /* argmin (cost, ordinal, step); cost = +inf when no record       */
    uint64_t reserved[6];         /* [0] plans admitted (have a valid first strategy), [1] plans handed from the
                                     bulk round to the chain kernel; rest 0                              */
} MetisSearchSummary;

/* Shard of the ordinal space evaluated by one call (multi-GPU: rank r of n, interleaved tiles). */
typedef struct MetisShard {
    int32_t rank;                 /* 0 <= rank < world                                              */
    int32_t world;
    int32_t tile;                 /* plans per interleave tile (multiple of 32)                     */
    int32_t reserved;             /* tuning: minimum number of admitted plans for which the bulk round (first
                                     partition attempt, one plan per thread) runs before the chain kernel;
                                     0 = default (12 x resident chain warps), INT32_MAX = chain kernel only */
} MetisShard;

const char *metis_last_error(void);
int metis_abi_version(void);

/*
 * Optional: CUDA events (cudaEvent_t as void*) that the NEXT metis_het_search call on this host
 * thread records immediately before and after its search kernel, so a caller can time that kernel
 * alone on the launching stream.  Pass NULLs to clear.
 */
void metis_set_profile_events(void *before_kernel, void *after_kernel);

/* Bytes of device scratch metis_het_search needs for a shard of `num_plans` plans: the packed tables
 * plus two lists of 16 B per plan (worst case: every plan has a valid strategy); `max_stage` is ignored.
 * metis_het_detail / metis_homo_cost need metis_het_workspace_bytes(problem, 0, 1). */
int64_t metis_het_workspace_bytes(const MetisProblem *problem, int64_t num_plans, int32_t max_stage);

/*
 * Replaces the loop of cost_het_cluster.py:24-48 for the shard's plans.
 *   records      [device] capacity MetisRecord slots (unordered; sort by (ordinal, step) to get
 *                estimate_costs order); may be NULL with capacity 0 when only the best is wanted
 *   detail       [device] optional, capacity * detail_stride bytes: per record
 *                dp code[num_stage], tp code[num_stage] (log2) then layer_partition[num_stage+1]
 *                (uint8 each); detail_stride >= 3*space->max_stage+1, or NULL
 *   workspace    [device] metis_het_workspace_bytes(problem, plans in shard, space->max_stage) bytes
 *   summary      [host]   filled asynchronously (use pinned memory)
 */
int metis_het_search(const MetisProblem *problem, const MetisPlanSpace *space, const MetisShard *shard,
                     MetisRecord *records, int64_t capacity, uint8_t *detail, int32_t detail_stride,
                     void *workspace, int64_t workspace_bytes, MetisSearchSummary *summary, void *stream);

/*
 * Re-evaluates the listed (ordinal, step) candidates and writes their strategies and
 * partition (same layout as `detail` above).  Used to materialise the winner / a ranked slice.
 *   picks [device] n MetisRecord (only ordinal and step are read)
 */
int metis_het_detail(const MetisProblem *problem, const MetisPlanSpace *space, const MetisRecord *picks,
                     int64_t n, uint8_t *detail, int32_t detail_stride, void *workspace,
                     int64_t workspace_bytes, void *stream);

/*
 * Verbose transcript (debug): replays the listed inter-stage plans, one thread each, and records the values the
 * reference prints while it evaluates them (search_space/plan.py:207-218, model/load_balancer.py:92,132-133,143,
 * model/cost_estimator.py:193,201-203,239-240, cost_het_cluster.py:43,48) as a stream of 64-bit words per plan; the
 * layout is documented in metis_b200/csrc/metis_trace.cuh and decoded by metis_b200/verbose.py.
 *   ordinals [device] n uint32 plan ordinals;  trace [device] n * words_per_plan uint64 (words_per_plan >= 64)
 */
int metis_het_trace(const MetisProblem *problem, const MetisPlanSpace *space, const uint32_t *ordinals, int64_t n,
                    uint64_t *trace, int32_t words_per_plan, void *workspace, int64_t workspace_bytes, void *stream);

/*
 * Replaces HomoCostEstimator.get_cost (model/cost_estimator.py:98-138) for n UniformPlans
 * (search_space/plan.py:12-18), as called from cost_homo_cluster.py:29.
 *   plans  [device] n x 5 int32 (dp, pp, tp, mbs, gbs)
 *   cost   [device] n doubles;  status [device] n int32: 0 ok, 1 KeyError (plan skipped), 2 oom flag set
 */
int metis_homo_cost(const MetisProblem *problem, int32_t type_id, const int32_t *plans, int64_t n,
                    double *cost, int32_t *status, void *workspace, int64_t workspace_bytes, void *stream);

/*
 * LayerComputeBalancer.run (model/load_balancer.py:197-207) for n independent instances.
 *   capa [device] n x stride doubles (stage capacities), num_stage [device] n int32,
 *   lc [device] norm_len doubles, partition [device] n x (stride+1) uint16 out (0xFFFF first = error),
 *   workspace [device] >= norm_len*8 + 256 bytes
 */
int metis_layer_balance(const double *capa, const int32_t *num_stage, int64_t n, int32_t stride,
                        const double *lc, int32_t norm_len, int32_t num_layers, uint16_t *partition,
                        void *workspace, int64_t workspace_bytes, void *stream);

/*
 * Orders the records written by metis_het_search on the device (stable LSD radix sort, one cooperative kernel).
 *   METIS_SORT_POSITION        by (ordinal, step): the order of `estimate_costs` as the reference appends it
 *                              (cost_het_cluster.py:44)
 *   METIS_SORT_RANKED          by (cost, ordinal, step): `sorted(estimate_costs, key=lambda kv: kv[-1])`
 *                              (cost_het_cluster.py:76; Python's sort is stable, so equal costs stay in
 *                              estimate_costs order)
 *   METIS_SORT_BY_COST_STABLE  by cost only, equal costs keep their current order (the second half of
 *                              METIS_SORT_RANKED, for records that are already in position order)
 *   records   [device] n records, sorted in place
 *   perm_out  [device] optional n uint32: perm_out[i] = index before the call of the record now at i
 *   workspace [device] metis_sort_workspace_bytes(n) bytes
 */
#define METIS_SORT_POSITION        0
#define METIS_SORT_RANKED          1
#define METIS_SORT_BY_COST_STABLE  2
int64_t metis_sort_workspace_bytes(int64_t n);
int metis_sort_records(MetisRecord *records, int64_t n, int32_t mode, uint32_t *perm_out, void *workspace,
                       int64_t workspace_bytes, void *stream);

/*
 * The min(k, n) first records of the METIS_SORT_RANKED order, without ordering all n (most-significant-digit radix
 * select over the (cost, ordinal, step) key, then metis_sort_records on the selected records only).  Records with
 * equal keys keep their input order, as in the sort.  k == 0 or n == 0 writes nothing.
 *   records   [device] n records in any order (read only)
 *   out       [device] min(k, n) records, ranked
 *   idx_out   [device] optional min(k, n) uint32: idx_out[i] = input position of out[i]
 *   workspace [device] metis_select_workspace_bytes(n, k) bytes
 */
int64_t metis_select_workspace_bytes(int64_t n, int64_t k);
int metis_select_records(const MetisRecord *records, int64_t n, int64_t k, MetisRecord *out, uint32_t *idx_out,
                         void *workspace, int64_t workspace_bytes, void *stream);

/*
 * Host-side enumeration of gen_dgroups_for_stages_with_variance (search_space/device_group.py:93-107)
 * in reference order.  Writes log2 codes, num_stages bytes per row, into out (host memory) and
 * returns the number of rows, or METIS_E_CAPACITY if capacity_rows is too small (call with
 * out == NULL to count).
 */
int64_t metis_enum_device_groups(int32_t num_stages, int32_t num_gpus, double variance,
                                 int32_t max_permute_len, uint8_t *out, int64_t capacity_rows);

/*
 * The same for every stage count first_stage..last_stage in one call, one host thread per stage count
 * (what InterStagePlanGenerator regenerates block by block, search_space/plan.py:130-142).  Tables are
 * written back to back into `out` (stage count s: rows_per_stage[s-first_stage] rows of s bytes).
 * Returns the total bytes (call with out == NULL to size the buffer; a second call with the buffer
 * recomputes the tables) or METIS_E_CAPACITY.
 */
int64_t metis_enum_device_group_tables(int32_t first_stage, int32_t last_stage, int32_t num_gpus,
                                       double variance, int32_t max_permute_len, int64_t *rows_per_stage,
                                       uint8_t *out, int64_t capacity_bytes);

/*
 * Device-side generation of the device-group rows (SURVEY.md 8(f)-1).  The host lists the compositions of every
 * stage count and merges their groups (search_space/device_group.py:7-81) - thousands of compositions - and the GPU
 * writes their multiset permutations in the reference's order (search_space/utils.py:72-88): millions of rows that
 * never exist on the host or on PCIe.  One record = one slice of at most METIS_COMP_SLICE_ROWS consecutive
 * permutations of one composition (the walk is sequential, so a warp skips to its slice and writes only that).
 */
typedef struct MetisCompRec {
    int64_t row_offset;           /* byte offset of the slice's first row in the row blob                      */
    uint32_t pool_offset;         /* the composition's entry in the pool: num_groups lengths, then `stages` log2
                                     codes of the groups in sorted order (utils.py:57)                         */
    uint16_t stages;
    uint16_t num_groups;          /* merged groups (<= METIS_MAX_PERMUTE_GROUPS on the device)                 */
    uint32_t first_row;           /* permutations of the composition before this slice                        */
    uint32_t num_rows;            /* permutations in this slice                                                */
} MetisCompRec;
#define METIS_COMP_SLICE_ROWS 64
#define METIS_MAX_PERMUTE_GROUPS 32
/* host: fills recs / pool (call with recs == NULL to size: returns the number of records, *pool_bytes the
 * pool size, *max_groups the largest num_groups); rows_per_stage like metis_enum_device_group_tables */
int64_t metis_enum_compositions(int32_t first_stage, int32_t last_stage, int32_t num_gpus, double variance,
                                int32_t max_permute_len, int64_t *rows_per_stage, MetisCompRec *recs,
                                int64_t recs_capacity, uint8_t *pool, int64_t pool_capacity, int64_t *pool_bytes,
                                int32_t *max_groups);
/* device: recs / pool [device], rows [device] receives every row (same layout as metis_enum_device_group_tables) */
int metis_generate_rows(const MetisCompRec *recs, int64_t num_comps, const uint8_t *pool, uint8_t *rows, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* METIS_B200_H */
