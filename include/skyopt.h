/*
 * skyopt.h -- C ABI of libskyopt, the B200 (sm_100a) placement-optimizer core.
 *
 * Nothing like this exists in the reference: SkyPilot's optimizer hot path is
 * pure Python / pandas. Each entry point below replaces the inner loop of the
 * reference function(s) cited next to it (paths relative to the SkyPilot
 * tree, commit 7808630). Callers bind it with ctypes (see INTEGRATION.md);
 * the signatures use plain pointers and sizes only.
 *
 * Ownership: the caller allocates every input and output buffer; the library
 * owns only device memory behind the opaque handle and keeps no caller
 * pointer after a call returns. Every function returns 0 on success and a
 * negative SKYOPT_E* code on failure; skyopt_last_error() returns the
 * thread-local message of the last failure. All calls are reentrant; a handle
 * is read-only after creation and may be shared by threads (each call borrows
 * a private stream + workspace from the handle's pool).
 */
#ifndef SKYOPT_H_
#define SKYOPT_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SKYOPT_ABI_VERSION 4

/* error codes */
#define SKYOPT_OK 0
#define SKYOPT_EINVAL (-1)   /* bad argument / malformed descriptor */
#define SKYOPT_ECUDA (-2)    /* CUDA runtime error (message has the detail) */
#define SKYOPT_ENOMEM (-3)   /* host or device allocation failed */
#define SKYOPT_ELIMIT (-4)   /* a documented capacity limit was exceeded */
#define SKYOPT_ENODEV (-5)   /* no usable CUDA device */

/* row flag bits (column `flags`, low byte); high byte = instance group id */
#define SKYOPT_F_VALID 0x0001u          /* real row (not alignment padding) */
#define SKYOPT_F_DEFAULT_FAMILY 0x0002u /* in the cloud's default CPU families
                                           (aws_catalog.py:37-65 etc.) */
#define SKYOPT_F_SSD 0x0004u            /* LocalDiskType == 'ssd' */
#define SKYOPT_F_NVME 0x0008u           /* NVMeSupported == True */
#define SKYOPT_F_HOST_FAMILY 0x0010u    /* GCP n1-* host VM families
                                           (gcp_catalog.py:73-77) */
#define SKYOPT_F_HAS_INSTANCE 0x0020u   /* InstanceType not NaN */
#define SKYOPT_F_PREMIUM_DISK 0x0040u   /* Azure S-series (azure.py:715-722) */

#define SKYOPT_NONE16 0xFFFFu
#define SKYOPT_ACC_SET_WORDS 32 /* accelerator-key bitmask: 1024 keys max */
#define SKYOPT_MAX_CLOUDS 32
#define SKYOPT_MAX_GROUP_ROWS 4096 /* rows of one instance type / acc key */

/*
 * Summary of 128 consecutive rows ("zone map" entry), computed at ingest:
 * the scan tests a query against it before touching the rows.
 */
typedef struct SkyoptZone {
  uint32_t flags_or;   /* OR of the low flag byte over the valid rows */
  uint32_t sig_lo;     /* bit (acc_key % 64) for every valid row's key ... */
  uint32_t sig_hi;     /* ... bits 32..63 */
  uint32_t groups;     /* bit (group % 32) for every valid row whose flags
                          high byte (GCP fixed-host group) is non-zero */
  uint64_t min_key[2]; /* cheapest 'Price' / 'SpotPrice' of the valid rows as
                          an order-preserving integer key (see
                          skyopt_price_key); all ones = none */
} SkyoptZone;

/*
 * The catalog as structure-of-arrays columns (host pointers; copied to HBM by
 * skyopt_catalog_create). Rows of all clouds are concatenated cloud by cloud
 * in original CSV order; each cloud's range is padded to a multiple of 128 rows
 * with flags == 0 rows. Replaces the pandas DataFrames of
 * sky/catalog/common.py:126-266 (LazyDataFrame / read_catalog).
 */
typedef struct SkyoptCatalogDesc {
  int64_t n_rows;            /* including padding rows */
  const double *price;       /* 'Price'      ; NaN = missing */
  const double *spot_price;  /* 'SpotPrice'  ; NaN = missing */
  const double *vcpus;       /* 'vCPUs'      ; NaN = missing */
  const double *mem;         /* 'MemoryGiB'  ; NaN = missing */
  const double *disk_total;  /* LocalDiskSize.fillna(0)*LocalDiskCount.fillna(0)
                                (common.py:499); may be NULL (all zero) */
  const uint16_t *acc_key;   /* id of (AcceleratorName, AcceleratorCount);
                                SKYOPT_NONE16 = no accelerator */
  const uint16_t *region_id; /* per-cloud rank of 'Region' in string order */
  const uint16_t *zone_id;   /* per-cloud rank of 'AvailabilityZone';
                                SKYOPT_NONE16 = missing */
  const uint16_t *flags;     /* SKYOPT_F_* | group << 8 */
  const int32_t *inst_id;    /* global instance-type id, -1 = NaN */
  int32_t n_clouds;
  int32_t n_inst;            /* instance types over all clouds */
  int32_t n_acc_keys;        /* <= 32 * SKYOPT_ACC_SET_WORDS */
  int32_t n_regions;         /* total over clouds */
  const int32_t *cloud_row_offsets;  /* [n_clouds+1], multiples of 128 */
  const int32_t *cloud_inst_offsets; /* [n_clouds+1] instance ids per cloud */
  const int32_t *cloud_region_offsets; /* [n_clouds+1] into region tables */
  const int32_t *cloud_n_zones;      /* [n_clouds]; 0 = cloud has no
                                        AvailabilityZone column */
  const uint8_t *region_is_us;       /* [n_regions] name.startswith('us-')
                                        (aws_catalog.py:327-336) */
  const int32_t *inst_row_offsets;   /* [n_inst+1] CSR into inst_rows */
  const int32_t *inst_rows;          /* row ids grouped by instance type,
                                        ascending inside a group */
  const int32_t *acc_row_offsets;    /* [n_acc_keys+1] CSR into acc_rows */
  const int32_t *acc_rows;           /* accelerator-only rows (inst_id < 0)
                                        grouped by acc_key (GCP) */
  const uint16_t *inst_acc_key;      /* [n_inst] acc_key of the type's first
                                        row (common.py:572-590) */
  const SkyoptZone *zone_map;        /* [n_rows / 128] static row summaries */
} SkyoptCatalogDesc;

/* comparison operators of a query */
#define SKYOPT_OP_NONE 0
#define SKYOPT_OP_EQ 1    /* ==            (common.py:452, :478) */
#define SKYOPT_OP_GE 2    /* >=  'n+'      (common.py:450, :474) */
#define SKYOPT_OP_RATIO 3 /* MemoryGiB >= vCPUs * r  'rx' (common.py:476) */
#define SKYOPT_DISK_NEAR 1 /* abs(total - size) < 1.0 (common.py:504) */
#define SKYOPT_DISK_GE 2   /* total >= size           (common.py:502) */

/* query flags */
#define SKYOPT_Q_ACC 0x1u    /* accelerator branch (common.py:641-694) */
#define SKYOPT_Q_FUZZY 0x2u  /* also collect the fuzzy table (:661-676) */
#define SKYOPT_Q_LIST 0x4u   /* also collect per-instance-type minima */
#define SKYOPT_Q_KEEP_NAN 0x8u /* list mode: NaN-price rows stay (no cap) */

/*
 * One catalog filter against one cloud's rows: the Resources-constraint
 * vector of get_instance_type_for_accelerator_impl (common.py:641-694) or
 * get_instance_type_for_cpus_mem_impl (common.py:518-569) after the per-cloud
 * wrappers (aws_catalog.py:249-319, gcp_catalog.py:282-393,
 * azure_catalog.py) turned their Python rules into flag / group requirements.
 */
typedef struct SkyoptQuery {
  int32_t cloud;        /* index into cloud_row_offsets */
  uint32_t qflags;      /* SKYOPT_Q_* */
  uint32_t flags_require; /* (row.flags & m) == m, low byte only */
  int32_t group;        /* required instance group id (high byte), 0 = any */
  int32_t acc_set;      /* exact-match accelerator-key set index, -1 = none */
  int32_t fuzzy_set;    /* fuzzy accelerator-key set index, -1 = none */
  int32_t price_col;    /* 0 'Price', 1 'SpotPrice' */
  int32_t cpus_op;      /* SKYOPT_OP_{NONE,EQ,GE} */
  int32_t mem_op;       /* SKYOPT_OP_{NONE,EQ,GE,RATIO} */
  int32_t disk_op;      /* 0, SKYOPT_DISK_NEAR, SKYOPT_DISK_GE */
  int32_t region_id;    /* per-cloud region id, -1 = any */
  int32_t zone_id;      /* per-cloud zone id, -1 = any */
  uint32_t flags_require2; /* like flags_require, but applied with the
                              cpus/memory stage (does not affect any_stage1):
                              Azure disk-tier drop in _make (azure.py:503-507) */
  int32_t pad_;
  double cpus;
  double mem;
  double disk_size;
  double max_price;     /* max_hourly_cost; +inf = none */
} SkyoptQuery;

/* result of one query */
typedef struct SkyoptScanResult {
  int32_t any_stage1;   /* a row matched accelerator+region/zone (stage 1 of
                           common.py:657-660); always 1 for CPU queries with
                           a match */
  int32_t best_row;     /* cheapest fully-matching row (lowest row id on a
                           price tie), -1 = none */
  int32_t best_inst;    /* its instance type id, -1 */
  int32_t n_list;       /* entries written to the list output */
  int32_t n_fuzzy;      /* entries written to the fuzzy output */
  int32_t pad_;
  double best_price;    /* NaN if none */
} SkyoptScanResult;

/*
 * One (requested Resources, cloud) slot of a task: which instance type to
 * expand into launchable (region[, zone]) candidates and how to cost them.
 * Replaces make_launchables_for_valid_region_zones (resources_utils.py:
 * 454-502), Cloud.regions_with_offering (aws.py:347-367, gcp.py:281-331),
 * common.get_region_zones (common.py:793-809) and the per-candidate
 * Resources.get_cost (resources.py:1685-1698; common.py:360-400,
 * gcp_catalog.py:424-442).
 */
typedef struct SkyoptSlot {
  int32_t cloud;
  int32_t query;        /* query whose cheapest row names the instance type;
                           -1 when inst_id is explicit */
  int32_t inst_id;      /* explicit instance type id; -1 = from query;
                           -2 = GCP 'TPU-VM' (no host rows, cost 0) */
  int32_t gate_query;   /* slot is empty unless this query's any_stage1 != 0
                           (GCP accelerator existence, gcp_catalog.py:352-357);
                           -1 = no gate */
  int32_t acc_set;      /* GCP: accelerator rows (exact count) to intersect
                           with the host VM zones; -1 = plain VM slot */
  int32_t price_col;    /* 0 on-demand, 1 spot */
  int32_t region_id;    /* exact request filter, -1 = any */
  int32_t zone_id;      /* exact request filter, -1 = any */
  int32_t split_by_zone; /* one candidate per zone (use_spot or
                            cloud.optimize_by_zone()) */
  int32_t us_first;     /* AWS / Lambda region order hack */
  int32_t cand_acc_key; /* accelerators of the launchable when they are not
                           implied by the instance type (GCP); -1 = derive
                           from inst_acc_key; used by the blocked filter */
  int32_t use_spot;     /* for the blocked filter */
  int32_t region_set;   /* allow-list of regions: index into acc_sets of a
                           bitmask over the cloud's region ids (bit r = region
                           r may be used), -1 = every region. Carries the
                           filters of Resources.get_valid_regions_for_launchable
                           (resources.py:1210-1246): the regions of a per-region
                           image_id dict and of a per-region ssh_proxy_command */
  int32_t pad_;
  double hours;         /* estimated_runtime / 3600 (optimizer.py:320-343) */
  double node_mult;     /* num_nodes; the device takes the reserved nodes of
                           each candidate off it (SkyoptReservation) */
  double time_value;    /* estimated_runtime, the TIME-mode value (:357) */
} SkyoptSlot;

/* Resources.should_be_blocked_by wildcard entry (resources.py:1938-1961) */
typedef struct SkyoptBlocked {
  int32_t cloud;     /* -1 = wildcard */
  int32_t inst_id;   /* -1 = wildcard, -2 = matches nothing */
  int32_t region_id; /* per-cloud id, -1 = wildcard, -2 = matches nothing */
  int32_t zone_id;   /* per-cloud id, -1 = wildcard, -2 = matches nothing */
  int32_t acc_key;   /* -1 = wildcard, -2 = matches nothing,
                        SKYOPT_NONE16 = "accelerators is None" never used */
  int32_t use_spot;  /* -1 = wildcard, 0 / 1 */
} SkyoptBlocked;

typedef struct SkyoptTask {
  int32_t slot_begin, slot_end; /* slots in candidate order
                                   (optimizer.py:1697-1732) */
  int32_t n_parents;
  int32_t parent_begin;         /* into the parents array (task indices local
                                   to the DAG); chain: one parent */
  int32_t edge_tariff_begin;    /* per parent: n_clouds doubles, egress value
                                   by the PARENT's cloud (optimizer.py:75-104,
                                   aws.py:667-688, gcp.py:395-404, ...) */
  int32_t src_tariff_begin;     /* n_clouds doubles by the candidate's cloud
                                   for a source task with inputs
                                   (optimizer.py:202-210); -1 = none */
} SkyoptTask;

typedef struct SkyoptDag {
  int32_t task_begin, task_end; /* topological order */
  int32_t is_chain;             /* 1: DP (optimizer.py:429-487); 0: exact
                                   search replacing the ILP (:490-637) */
  int32_t minimize_cost;        /* 1 COST, 0 TIME */
  int32_t blocked_begin, blocked_end;
} SkyoptDag;

/* one launchable candidate as the optimizer sees it */
typedef struct SkyoptCandidate {
  int32_t slot;       /* global slot index */
  int32_t inst_id;
  int32_t region_id;  /* per-cloud id */
  int32_t zone_id;    /* per-cloud id, -1 = region-level candidate */
  double hourly;      /* instance (+ accelerator) hourly price */
  double value;       /* cost or time entering the DP (optimizer.py:353-357) */
} SkyoptCandidate;

typedef struct SkyoptDagResult {
  int32_t status;     /* 0 ok; 1 = a task has no candidate (first such task
                         in task_fail); 2 = general DAG beyond the device
                         enumeration (more than 16 tasks or 2^26 cloud
                         assignments): the caller solves it from the candidate
                         tables (skypilot_b200/dag_solver.py, exact bucket
                         elimination for the COST objective) */
  int32_t task_fail;
  double objective;   /* best_total_objective */
} SkyoptDagResult;

/*
 * Consumable reserved capacity of one (cloud, instance type, zone): the sum
 * over the reservations that the candidate may use
 * (Resources.get_reservations_available_resources, resources.py:1785-1812;
 * aws.py:1490-1519, gcp.py:1419-1438). A COST-objective, non-spot candidate
 * with a zone is valued hourly * hours * max(num_nodes - available, 0)
 * (optimizer.py:344-354). The table is sorted by (cloud, inst_id, zone_id)
 * and has no duplicate keys.
 */
typedef struct SkyoptReservation {
  int32_t cloud, inst_id, zone_id;  /* same ids as SkyoptCandidate / SkyoptBlocked */
  int32_t available;                /* consumable reserved nodes, summed, > 0 */
} SkyoptReservation;

typedef struct SkyoptProblem {
  const SkyoptQuery *queries;
  int32_t n_queries;
  const uint32_t *acc_sets; /* [n_acc_sets][SKYOPT_ACC_SET_WORDS] */
  int32_t n_acc_sets;
  const SkyoptSlot *slots;
  int32_t n_slots;
  const SkyoptTask *tasks;
  int32_t n_tasks;
  const int32_t *parents;
  int32_t n_parents;
  const double *tariffs;
  int32_t n_tariffs;
  const SkyoptBlocked *blocked;
  int32_t n_blocked;
  const SkyoptDag *dags;
  int32_t n_dags;
  const SkyoptReservation *reservations; /* may be NULL when n_reservations == 0 */
  int32_t n_reservations;
} SkyoptProblem;

typedef struct SkyoptSolution {
  SkyoptScanResult *scan;      /* [n_queries] or NULL */
  int32_t *slot_count;         /* [n_slots] candidates before blocking, or NULL */
  int32_t *slot_inst;          /* [n_slots] instance type expanded, or NULL */
  SkyoptCandidate *chosen;     /* [n_tasks] the plan */
  int32_t *chosen_index;       /* [n_tasks] index in the task's candidate list */
  int32_t *task_n_candidates;  /* [n_tasks] after the blocked filter */
  SkyoptDagResult *dag;        /* [n_dags] */
  SkyoptCandidate *candidates; /* optional full tables, capacity cand_cap */
  int64_t cand_cap;            /* 0 = do not return the tables */
  int64_t *task_cand_offset;   /* [n_tasks+1] into candidates, or NULL */
} SkyoptSolution;

typedef struct SkyoptStats {
  float scan_ms;   /* device time of the filter+argmin scan (CUDA events) */
  float expand_ms; /* region/zone expansion + cost */
  float solve_ms;  /* blocked filter + DP / exact search */
  float total_ms;  /* first H2D to last D2H */
  int32_t scan_launches;
  int32_t total_launches;
  int64_t scan_rows;       /* sum over queries of rows scanned */
  int64_t scan_passes_rows; /* rows streamed from HBM (queries fused per pass) */
  float scan_kernel_ms;     /* the scan kernel launch alone (events around it) */
  int32_t scan_blocks;      /* its grid size */
  int32_t scan_form;        /* which scan kernel ran: 0 one tile per block,
                               1 streaming (TMA), 2 queue form, 3 class-table
                               scan (scan2_kernel), 4 the same inside the fused
                               step_kernel */
  int32_t reserved_;        /* scan_form >= 3: rows streamed by the launch in
                               the 10-byte layout (one pass per query group) */
} SkyoptStats;

typedef struct SkyoptCatalog SkyoptCatalog; /* opaque */

int skyopt_abi_version(void);
/* Order-preserving map double -> uint64 used for prices (NaN excluded). */
uint64_t skyopt_price_key(double price);
const char *skyopt_last_error(void);
int skyopt_device_count(int *count);

/* replaces read_catalog / LazyDataFrame (common.py:126-266): upload once */
int skyopt_catalog_create(const SkyoptCatalogDesc *desc, int device,
                          SkyoptCatalog **out);
int skyopt_catalog_destroy(SkyoptCatalog *cat);
int skyopt_catalog_bytes(const SkyoptCatalog *cat, int64_t *device_bytes,
                         int64_t *row_bytes);
/* Kernel selection: 0 = auto -- the class-table scan inside ONE cooperative
 * launch per step (scan2 -> barrier -> place -> chain DP) when the catalog's
 * class dictionaries fit shared memory and the problem has no list / fuzzy
 * queries, else the round-1 kernels picked by the amount of work (queue form
 * for large scans, one tile per block for small ones). Forced: 1 = one tile per
 * block, 2 / 3 = TMA streaming kernel (3: three tiles per block), 4 = queue
 * form, 5 = queue form with 32 tiles per block, 6 = class-table scan (fused),
 * 7 = 6 with the zone map and the running bound ignored (HBM stress: every row
 * is streamed and scored), 8 = 6 as separate launches (scan2, place, solve),
 * 9 = 8 without pruning. Results are identical in every mode; used by tests,
 * tuning and the roofline measurement. SKYOPT_SCAN_MODE=tile|stream|stream3|
 * queue|queue32|fast|fast-noprune|fast-split|fast-split-noprune sets the
 * default. */
int skyopt_catalog_set_scan_mode(SkyoptCatalog *cat, int mode);

/*
 * Filter + argmin only: get_instance_type_for_accelerator_impl /
 * get_instance_type_for_cpus_mem_impl (common.py:518-569, :641-694) for a
 * batch of queries. list_out / fuzzy_out may be NULL; otherwise they receive,
 * per query, up to list_cap (instance id, min price) / fuzzy_cap (acc key,
 * min Price) pairs sorted by price.
 */
int skyopt_scan(SkyoptCatalog *cat, const SkyoptQuery *queries, int n_queries,
                const uint32_t *acc_sets, int n_acc_sets,
                SkyoptScanResult *results, int32_t *list_ids,
                double *list_prices, int list_cap, int32_t *fuzzy_keys,
                double *fuzzy_prices, int fuzzy_cap, SkyoptStats *stats);

/*
 * Cheapest offering per group for accelerator listings: the reduction inside
 * list_accelerators_impl (sky/catalog/common.py:756-768,
 * sort_values(['Price', 'SpotPrice'[, 'Region']]).drop_duplicates(keep=
 * 'first')). group_ids are global instance-type ids (by_acc_key == 0) or
 * accelerator-key ids (by_acc_key != 0: GCP's accelerator-only rows,
 * gcp_catalog.py:445-571) of `cloud`. region_mask (may be NULL = every region)
 * has one bit per region of the cloud (local region id). out_rows receives,
 * per group, the catalog row of the winner -- or, with per_region, one row
 * per region of the cloud ([n_groups][n_regions_of_cloud]); -1 = no row.
 */
int skyopt_list_offerings(SkyoptCatalog *cat, int cloud, int by_acc_key,
                          const int32_t *group_ids, int n_groups,
                          const uint32_t *region_mask, int per_region,
                          int32_t *out_rows);

/*
 * The fused hot path: Optimizer._optimize_dag (optimizer.py:1381-1512) for a
 * batch of independent DAGs -- scan, expansion, cost, blocked filter and
 * chain DP / exact DAG search stay on the device; one H2D and one D2H copy.
 */
int skyopt_optimize(SkyoptCatalog *cat, const SkyoptProblem *problem,
                    SkyoptSolution *solution, SkyoptStats *stats);

/*
 * DP / exact search alone, on candidate tables the caller already has:
 * Optimizer._optimize_by_dp (optimizer.py:429-487) and _optimize_by_ilp
 * (:490-637) as stand-alone operators. Task t's candidates are
 * values[task_offsets[t] .. task_offsets[t+1]) (cost or time entering the
 * objective, in the reference's dictionary order) with their cloud index in
 * `clouds`; tasks / parents / tariffs / dags as in SkyoptProblem (slot fields
 * of the tasks are ignored). Writes the chosen candidate index per task.
 */
int skyopt_solve_tables(SkyoptCatalog *cat, const double *values,
                        const int32_t *clouds, const int64_t *task_offsets,
                        const SkyoptTask *tasks, int n_tasks,
                        const int32_t *parents, int n_parents,
                        const double *tariffs, int n_tariffs,
                        const SkyoptDag *dags, int n_dags,
                        int32_t *chosen_index, SkyoptDagResult *results);

/*
 * Failover re-optimisation (the provisioner's retry loop,
 * sky/backends/cloud_vm_ray_backend.py:332-339, :1817-1825: every failed launch
 * adds a wildcard to blocked_resources and calls Optimizer.optimize again).
 * A session runs skyopt_optimize once and keeps the expanded candidate sets
 * of its DAGs resident on the device; skyopt_session_resolve then only
 * uploads a new blocked list (applied to every DAG of the session), re-runs
 * the blocked filter + cost kernel and the solver, and reads the plan back --
 * no catalog scan, no region/zone expansion. The session owns a private
 * stream and workspace until it is closed; `problem`'s own blocked entries
 * are the list of the first solve.
 */
typedef struct SkyoptSession SkyoptSession;
int skyopt_session_open(SkyoptCatalog *cat, const SkyoptProblem *problem,
                        SkyoptSolution *solution, SkyoptStats *stats,
                        SkyoptSession **out);
int skyopt_session_resolve(SkyoptSession *session, const SkyoptBlocked *blocked,
                           int n_blocked, SkyoptSolution *solution,
                           SkyoptStats *stats);
void skyopt_session_close(SkyoptSession *session);

/*
 * Device-resident timing loop for bench.py: uploads `problem` once, then runs
 * the kernels `iters` times, flushing L2 (writing a buffer > 126 MB) before
 * every iteration when flush_l2 != 0; per-iteration device times (CUDA
 * events around the kernels only) are written to iter_ms[iters] and the
 * duration of the scan kernel launch alone to scan_kernel_ms[iters].
 */
int skyopt_optimize_timed(SkyoptCatalog *cat, const SkyoptProblem *problem,
                          SkyoptSolution *solution, int iters, int flush_l2,
                          float *iter_ms, float *scan_kernel_ms,
                          SkyoptStats *stats);

#ifdef __cplusplus
}
#endif
#endif /* SKYOPT_H_ */
