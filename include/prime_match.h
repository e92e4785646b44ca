/*
 * prime_match.h — C ABI of the B200-native task<->worker matching engine.
 *
 * Drop-in boundary for the Prime Protocol orchestrator's scheduling hot path.
 * Every entry point below names the reference interface (file:line under the
 * reference checkout, crates/...) that it replaces or feeds.  Plain pointers
 * and sizes only; no C++/torch types cross this boundary.  All functions
 * return 0 (PM_OK) or a negative pm_status, never unwind, never abort
 * (reference error convention: failures are swallowed to an empty answer and
 * retried next tick — crates/orchestrator/src/plugins/node_groups/
 * scheduler_impl.rs:24-30,86-104 and mod.rs:188-194).
 *
 * Vocabulary follows the reference: worker == OrchestratorNode
 * (crates/orchestrator/src/models/node.rs:10-37), ask == one
 * NodeGroupConfiguration row {min,max,ComputeRequirements}
 * (crates/orchestrator/src/plugins/node_groups/mod.rs:30-37), evaluation ==
 * one is_node_compatible_with_config call (mod.rs:206-215).
 */
#ifndef PRIME_MATCH_H
#define PRIME_MATCH_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PM_ABI_VERSION 1u
#define PM_NONE 0xFFFFFFFFu
#define PM_COST_INF INT64_MAX

typedef enum pm_status {
  PM_OK = 0,
  PM_E_INVALID = -1,     /* bad argument / table shape                        */
  PM_E_CUDA = -2,        /* CUDA runtime error; text in pm_last_error         */
  PM_E_NO_DEVICE = -3,   /* no sm_100 device visible: the engine never falls  */
                         /* back to a CPU path                                */
  PM_E_STATE = -4,       /* call order violated (e.g. match before tables)    */
  PM_E_NOMEM = -5,
  PM_E_UNSUPPORTED = -6,
  PM_E_PARSE = -7        /* requirement string rejected (node.rs:180-374)     */
} pm_status;

/* ------------------------------------------------------------------------ */
/* Worker table: SoA mirror of OrchestratorNode + ComputeSpecs               */
/* (crates/shared/src/models/node.rs:25-35,72-78,153-157).  Two 16-byte      */
/* planes so that one worker is exactly two coalesced 128-bit loads.         */
/* ------------------------------------------------------------------------ */
enum pm_worker_flag {
  PM_W_HEALTHY        = 1u << 0,  /* status == NodeStatus::Healthy  (mod.rs:494) */
  PM_W_P2P            = 1u << 1,  /* p2p_id.is_some()               (mod.rs:495) */
  PM_W_ASSIGNED       = 1u << 2,  /* present in node_to_group       (mod.rs:496) */
  PM_W_HAS_SPECS      = 1u << 3,  /* compute_specs.is_some()                     */
  PM_W_HAS_GPU        = 1u << 4,  /* specs.gpu.is_some()                         */
  PM_W_HAS_GPU_COUNT  = 1u << 5,
  PM_W_HAS_GPU_MEM    = 1u << 6,
  PM_W_HAS_GPU_MODEL  = 1u << 7,
  PM_W_HAS_CPU        = 1u << 8,  /* specs.cpu.is_some()                         */
  PM_W_HAS_CPU_CORES  = 1u << 9,
  PM_W_HAS_RAM        = 1u << 10,
  PM_W_HAS_STORAGE    = 1u << 11,
  PM_W_HAS_LOC        = 1u << 12  /* location.is_some()                          */
};

typedef struct pm_worker_a {   /* plane A, 16 B */
  uint32_t gpu_count;          /* GpuSpecs.count      */
  uint32_t gpu_mem_mb;         /* GpuSpecs.memory_mb  */
  uint32_t model_id;           /* interned GpuSpecs.model (pm_intern_model); must be < n_models of the model table in */
                               /* force when PM_W_HAS_GPU_MODEL is set (a precondition: the kernels index the table by it) */
  uint32_t flags;              /* pm_worker_flag bits */
} pm_worker_a;

typedef struct pm_worker_b {   /* plane B, 16 B */
  uint32_t cpu_cores;          /* CpuSpecs.cores */
  uint32_t ram_mb;
  uint32_t storage_gb;
  uint32_t ext_ask_price;      /* north-star extension column; 0 when unused */
} pm_worker_b;

/* ------------------------------------------------------------------------ */
/* Ask table: one row per enabled NodeGroupConfiguration in PRIORITY ORDER   */
/* (mod.rs:150-164 then :399-418; pm_sort_configs reproduces it), plus a     */
/* CSR list of GpuRequirements OR-options (node.rs:58-70).                   */
/* ------------------------------------------------------------------------ */
enum pm_ask_flag {
  PM_A_HAS_REQ        = 1u << 0,  /* compute_requirements.is_some()  (mod.rs:210-214) */
  PM_A_REQ_CPU        = 1u << 1,  /* requirements.cpu.is_some()      (node.rs:381)    */
  PM_A_REQ_CPU_CORES  = 1u << 2,  /* requirements.cpu.cores.is_some  (node.rs:533)    */
  PM_A_REQ_RAM        = 1u << 3,
  PM_A_REQ_STORAGE    = 1u << 4
};

typedef struct pm_ask {        /* 32 B */
  uint32_t flags;              /* pm_ask_flag bits */
  uint32_t n_opts;             /* requirements.gpu.len() */
  uint32_t opt_off;            /* first pm_gpu_opt of this ask */
  uint32_t cpu_cores;
  uint32_t ram_mb;
  uint32_t storage_gb;
  uint32_t min_group_size;
  uint32_t max_group_size;
} pm_ask;

enum pm_opt_present {
  PM_O_COUNT   = 1u << 0,
  PM_O_MODEL   = 1u << 1,
  PM_O_MEM     = 1u << 2,   /* memory_mb        */
  PM_O_MEM_MIN = 1u << 3,   /* memory_mb_min    */
  PM_O_MEM_MAX = 1u << 4,   /* memory_mb_max    */
  PM_O_TOT_MIN = 1u << 5,   /* total_memory_min */
  PM_O_TOT_MAX = 1u << 6    /* total_memory_max */
};

typedef struct pm_gpu_opt {    /* 32 B; field-for-field GpuRequirements */
  uint32_t present;            /* pm_opt_present bits */
  uint32_t count;
  uint32_t memory_mb;
  uint32_t memory_mb_min;
  uint32_t memory_mb_max;
  uint32_t total_memory_min;
  uint32_t total_memory_max;
  uint32_t pattern_id;         /* interned requirement model list (pm_intern_pattern) */
} pm_gpu_opt;

/* ------------------------------------------------------------------------ */
/* Host-side model-string interning.  The substring predicate of            */
/* GpuSpecs::meets (node.rs:463-484) is evaluated once per distinct          */
/* (requirement pattern, worker model) pair on the host and shipped to the   */
/* device as a bit table; per (ask, worker) pair the device does one bit     */
/* test.  No GPU needed for these calls.                                     */
/* ------------------------------------------------------------------------ */
typedef struct pm_interner pm_interner;
pm_interner* pm_interner_create(void);
void         pm_interner_destroy(pm_interner*);
uint32_t     pm_intern_model(pm_interner*, const char* spec_model);      /* worker side */
uint32_t     pm_intern_pattern(pm_interner*, const char* req_model);     /* ask side    */
/* bits[p * words + (m >> 5)] >> (m & 31) & 1  <=>  pattern p accepts model m;  */
/* words = ceil(n_models / 32).  Pointer is valid until the next intern call.   */
int pm_interner_table(pm_interner*, const uint32_t** bits, uint32_t* n_patterns,
                      uint32_t* n_models, uint32_t* words_per_pattern);

/* ComputeRequirements::from_str (node.rs:180-374).  Fills *ask (flags, n_opts,
 * cpu/ram/storage; opt_off/min/max untouched) and up to max_opts options.   */
int pm_parse_requirements(const char* s, pm_interner* interner, pm_ask* ask,
                          pm_gpu_opt* opts, uint32_t max_opts, uint32_t* n_opts,
                          char* err, size_t err_len);

/* NodeGroupsPlugin::new_with_policy sort (mod.rs:150-164): stable, by
 * min_group_size desc, then with-requirements before without.  perm_out[i] =
 * index of the config that lands at priority i.                             */
int pm_sort_configs(const uint32_t* min_group_size, const uint8_t* has_requirements,
                    uint32_t n, uint32_t* perm_out);

/* Node ids.  The reference parses every wire id (`node.id.parse::<Address>()`, discovery/monitor.rs:240) and uses
 * `Address::to_string()` — "0x" + 40 hex digits in EIP-55 checksum case (alloy-primitives 1.1.0, Cargo.lock) — as the
 * key of every store, of node_to_group and of the BTreeSet that decides GROUP_INDEX (mod.rs:63-69,424-434).
 * pm_address_canonical does the same for a C string: accepts 40 hex digits with or without "0x", any case (no
 * checksum validation, like Address::from_str), writes the 42-character checksummed form + NUL.  PM_E_INVALID otherwise. */
int pm_address_canonical(const char* address, char out[43]);

/* ------------------------------------------------------------------------ */
/* Engine                                                                     */
/* ------------------------------------------------------------------------ */
typedef struct pm_engine pm_engine;

enum pm_cfg_flag {
  PM_CFG_TIMING = 1u << 0     /* record CUDA events per kernel class (pm_stats.ms_*) */
};

typedef struct pm_cfg {
  uint32_t abi_version;        /* PM_ABI_VERSION */
  int32_t  device;             /* CUDA ordinal */
  uint32_t flags;              /* pm_cfg_flag */
  uint32_t reserved0;
  uint64_t cost_tile_bytes;    /* HBM budget for one materialised cost tile; 0 = 8 GiB */
  /* Worker sharding across GPUs (SURVEY 8e): this engine evaluates the        */
  /* contiguous canonical-order range [shard_first, shard_first+shard_count)   */
  /* of the global worker table; shard_count == 0 means "all".                 */
  uint32_t shard_first;
  uint32_t shard_count;
  void*    stream;             /* cudaStream_t to launch on (e.g. the caller's torch     */
                               /* stream, so its CUDA events bracket the kernels);        */
                               /* NULL = the engine creates a private non-blocking stream */
} pm_cfg;

int         pm_create(const pm_cfg* cfg, pm_engine** out);
void        pm_destroy(pm_engine*);
const char* pm_last_error(const pm_engine*);   /* NULL engine -> last create error */

/* Pinned host memory for the caller-owned tables (SURVEY 8b "ownership").   */
void* pm_alloc_pinned(size_t bytes);
void  pm_free_pinned(void*);

/* replaces the per-pass TaskStore/config reads (mod.rs:399-418)             */
/* [opt_off, opt_off + n_opts) ranges may overlap or be shared between asks.  */
int pm_set_asks(pm_engine*, const pm_ask* asks, uint32_t n_asks,
                const pm_gpu_opt* opts, uint32_t n_opts);
int pm_set_model_table(pm_engine*, const uint32_t* bits, uint32_t n_patterns,
                       uint32_t n_models, uint32_t words_per_pattern);
/* replaces NodeStore::get_nodes per pass (store/domains/node_store.rs:163-209);
 * row index == canonical order (SURVEY 8c determinisation rule 1).          */
int pm_set_worker_count(pm_engine*, uint32_t n_workers);
int pm_upsert_workers(pm_engine*, const pm_worker_a* a, const pm_worker_b* b,
                      uint32_t first, uint32_t n);
/* NodeLocation.latitude/longitude (node.rs:543-550); only read in proximity mode */
int pm_set_worker_locations(pm_engine*, const double* lat, const double* lon,
                            uint32_t first, uint32_t n);
/* rank of the worker's address string in BTreeSet<String> order
 * (mod.rs:63-69,424-434); decides member order inside a group               */
int pm_set_worker_addr_rank(pm_engine*, const uint32_t* rank, uint32_t first, uint32_t n);
/* status / assigned deltas (status_update_impl.rs:8-39, mod.rs:1423-1487)   */
int pm_set_flags(pm_engine*, const uint32_t* idx, const uint32_t* flags, uint32_t n);

/* Resident tables with deltas: a long-running host keeps the worker table on the device between management passes and
 * sends only the rows that changed (status / assigned / specs / location), instead of NodeStore::get_nodes' full
 * read per pass (store/domains/node_store.rs:163-209).
 *   pm_resize_workers   grow (or shrink) the table, keeping the rows it holds; new rows are empty (no candidate)
 *   pm_update_workers   scatter n rows by index; lat/lon both NULL or both given
 *   pm_table_version    changes whenever any table call ran: lets a caller detect that someone else used the engine
 *   pm_create_sibling   a second engine on the same device with the same configuration (own stream and tables)   */
int      pm_resize_workers(pm_engine*, uint32_t n_workers);
int      pm_update_workers(pm_engine*, const uint32_t* idx, const pm_worker_a* a, const pm_worker_b* b,
                           const double* lat, const double* lon, uint32_t n);
uint64_t pm_table_version(const pm_engine*);
int      pm_create_sibling(const pm_engine*, pm_engine** out);

/* NORTH-STAR EXTENSION columns (no reference counterpart; only PM_MODE_AUCTION reads them):
 * per-ask price cap against pm_worker_b.ext_ask_price, and the auction's parameters
 * (value = -(ask_price * cost_scale) - price; eps runs eps_start, /eps_div, ..., 1).       */
int pm_set_ask_price_caps(pm_engine*, const uint32_t* price_cap, uint32_t n_asks);
int pm_set_auction_params(pm_engine*, uint64_t cost_scale, uint64_t eps_start, uint32_t eps_div);
/* `reputation` (north_star worker column; SURVEY 8 A21 side column ext_reputation:u32) and the per-ask floor on it:
 *   feasible(t,w) additionally requires reputation[w] >= min_reputation[t]   (PM_MODE_AUCTION only).
 * Both default to 0 (no clause).  The worker column follows the worker table: pm_resize_workers keeps it,
 * pm_set_worker_count drops it.  min_reputation is per ask, after pm_set_asks, like the price caps.      */
int pm_set_worker_reputation(pm_engine*, const uint32_t* reputation, uint32_t first, uint32_t n);
int pm_set_ask_min_reputation(pm_engine*, const uint32_t* min_reputation, uint32_t n_asks);

enum pm_mode {
  PM_MODE_FIRST_FIT = 0,   /* try_form_new_groups, ProximityOptimizationPolicy{enabled:false} */
  PM_MODE_PROXIMITY = 1,   /* ... {enabled:true}  (mod.rs:524-552), the reference default     */
  PM_MODE_PROXIMITY_MERGE = 3, /* try_merge_solo_groups' batch selection (mod.rs:752-848) over a table that  */
                           /* holds only the nodes of solo groups, in get_all_groups() order               */
  PM_MODE_AUCTION   = 2    /* north-star extension: price-capped forward auction, one worker  */
                           /* per ask (pm_auction.cuh); no reference counterpart, self-oracle */
};
enum pm_path {
  PM_PATH_MATERIALIZED = 0,      /* build a cost tile in HBM, then argmin over it: 16-bit price words when every */
                                 /* ext_ask_price <= 0xFFFE and the fast predicate applies, else int64 keys    */
  PM_PATH_FUSED        = 1u << 8,/* evaluate + reduce on chip, matrix never written   */
  PM_NO_ASK_STATS      = 1u << 9 /* with PM_PATH_FUSED: skip ask_best / ask_count (the reference modes only
                                    need the per-worker first feasible ask); they read INF / 0 then      */
};

typedef struct pm_stats {
  uint64_t evals;            /* predicate evaluations executed on the device        */
  uint64_t cost_bytes_written; /* materialised path: 2 (16-bit tile) or 8 (int64 tile) B per evaluation */
  uint64_t cost_bytes_read;
  uint32_t n_tiles;          /* cost tiles; auction mode: class (re)scans           */
  uint32_t n_launches;       /* kernels of this library launched by the last match  */
  uint32_t n_bumped;         /* workers displaced by an under-filled tail group     */
  uint32_t n_rounds;         /* auction rounds (extension mode)                     */
  float ms_build;            /* sum over launches, CUDA events on the engine stream */
  float ms_argmin;
  float ms_fused;
  float ms_resolve;
  float ms_total;
  uint32_t n_build_launches; /* auction mode: class pool refills                    */
  uint32_t n_argmin_launches;
  uint32_t n_fused_launches; /* auction mode: per-ask fallback scans                */
  float    ms_exchange;      /* sharded pass: pack + all-gather + fold, on the engine stream */
  uint64_t exchange_bytes;   /* bytes this rank received in the exchange            */
} pm_stats;

typedef struct pm_result {
  uint32_t n_workers;
  uint32_t n_asks;
  uint32_t n_groups;
  uint32_t n_members;
  /* all arrays are engine-owned pinned host memory, valid until the next
   * pm_fetch_result / pm_destroy on this engine                             */
  const uint32_t* worker_group;   /* [n_workers] group index or PM_NONE                 */
  const uint32_t* worker_ask;     /* [n_workers] ask (config) index or PM_NONE          */
  const uint32_t* group_ask;      /* [n_groups]  configuration of the group             */
  const uint32_t* group_off;      /* [n_groups+1] CSR offsets into group_members        */
  const uint32_t* group_members;  /* worker indices, BTreeSet (addr_rank) order         */
  const int64_t*  ask_best;       /* [n_asks] row argmin: cost<<32 | worker, PM_COST_INF */
  const uint32_t* ask_count;      /* [n_asks] feasible candidate workers of the ask      */
  pm_stats stats;
} pm_result;

/* The management pass (replaces try_form_new_groups, mod.rs:478-628).
 * mode = pm_mode | pm_path.  Device compute only: tables must be resident.  */
int pm_match(pm_engine*, uint32_t mode);
/* D2H of the last match into engine-owned pinned buffers.                   */
int pm_fetch_result(pm_engine*, pm_result* out);
int pm_get_stats(const pm_engine*, pm_stats* out);
/* Build the cost rows of asks [t0, t0+nt) against this engine's worker range and
 * copy them to host_out[nt * n_cols] (row-major, n_cols = shard width): the
 * materialised matrix itself, for external solvers and for bit-exact checks.  */
int pm_build_cost_tile(pm_engine*, uint32_t t0, uint32_t nt, int64_t* host_out);

/* Multi-GPU plumbing (SURVEY 8e): between pm_match_local and pm_match_finish
 * the host all-reduces/all-gathers these device buffers with NCCL.          */
enum pm_buffer {
  PM_BUF_WORKER_FIRST_ASK = 0,  /* uint32[n_workers] global; only the shard range is written */
  PM_BUF_ASK_BEST         = 1,  /* int64 [n_asks] packed row argmin (allreduce MIN)          */
  PM_BUF_ASK_COUNT        = 2   /* uint32[n_asks] (allreduce SUM)                            */
};
/* Re-target the engine at the range [first, first+count) of the worker table (count 0 = to the end). */
int pm_set_shard(pm_engine*, uint32_t first, uint32_t count);
int pm_match_local(pm_engine*, uint32_t mode);    /* evaluation over this shard only */
int pm_match_finish(pm_engine*, uint32_t mode);   /* resolution sweep over the global arrays */
int pm_device_buffer(pm_engine*, uint32_t which, void** dev_ptr, size_t* bytes);
int pm_stream_sync(pm_engine*);

/* ------------------------------------------------------------------------ */
/* Multi-GPU inside the engine (SURVEY 8b "multi-GPU is inside the engine", 8e).  */
/* The path shards by workers: every GPU evaluates all asks against an equal     */
/* contiguous share of the canonical worker order; ONE packed all-gather per     */
/* pass (NCCL over NVLink, resolved at run time) carries {per-ask (min cost,     */
/* argmin) + feasible count, per-worker first feasible ask}; every GPU then runs */
/* the same O(W+T) resolution sweep on identical arrays.  With a communicator    */
/* attached pm_match does all of it; the shard is the rank's share.              */
/* ------------------------------------------------------------------------ */
typedef struct pm_comm pm_comm;
#define PM_COMM_ID_BYTES 128
/* one process per GPU: rank 0 makes the id, the host hands it to every rank (any transport) */
int  pm_comm_unique_id(uint8_t id_out[PM_COMM_ID_BYTES]);
int  pm_comm_create(const uint8_t unique_id[PM_COMM_ID_BYTES], uint32_t n_ranks, uint32_t rank, int32_t device,
                    pm_comm** out);
void pm_comm_destroy(pm_comm*);
int  pm_attach_comm(pm_engine*, pm_comm*);   /* NULL detaches; the communicator must outlive the engine's use of it */

/* One process, several GPUs — the form the orchestrator's single management loop                          */
/* (crates/orchestrator/src/main.rs:283-289, mod.rs:180-203) calls: table calls go to every device,        */
/* pm_multi_match is one sharded pass, the result is read from device 0.  cfg->device/shard/stream ignored. */
typedef struct pm_multi pm_multi;
int         pm_multi_create(const pm_cfg* cfg, const int32_t* devices, uint32_t n_devices, pm_multi** out);
void        pm_multi_destroy(pm_multi*);
uint32_t    pm_multi_size(const pm_multi*);
pm_engine*  pm_multi_engine(pm_multi*, uint32_t i);   /* per-device access (stats, auction params, ...) */
const char* pm_multi_last_error(const pm_multi*);
int pm_multi_set_asks(pm_multi*, const pm_ask* asks, uint32_t n_asks, const pm_gpu_opt* opts, uint32_t n_opts);
int pm_multi_set_model_table(pm_multi*, const uint32_t* bits, uint32_t n_patterns, uint32_t n_models,
                             uint32_t words_per_pattern);
int pm_multi_set_worker_count(pm_multi*, uint32_t n_workers);
int pm_multi_upsert_workers(pm_multi*, const pm_worker_a* a, const pm_worker_b* b, uint32_t first, uint32_t n);
int pm_multi_set_worker_locations(pm_multi*, const double* lat, const double* lon, uint32_t first, uint32_t n);
int pm_multi_set_worker_addr_rank(pm_multi*, const uint32_t* rank, uint32_t first, uint32_t n);
int pm_multi_set_flags(pm_multi*, const uint32_t* idx, const uint32_t* flags, uint32_t n);
int pm_multi_sync(pm_multi*);
int pm_multi_match(pm_multi*, uint32_t mode);
int pm_multi_fetch_result(pm_multi*, pm_result* out);

uint32_t pm_abi_version(void);

/* ------------------------------------------------------------------------ */
/* Host mirror of the reference's plugin interface for this path              */
/* (protocol_b200/csrc/pm_plugin.cpp).  In-process tables replace Redis; group */
/* formation always runs on the engine (no CPU evaluation path).              */
/* ------------------------------------------------------------------------ */
typedef struct pm_plugin pm_plugin;

typedef struct pm_plugin_policy {     /* mod.rs:71-98 */
  uint8_t task_switching_enabled;     /* TaskSwitchingPolicy.enabled               */
  uint8_t prefer_larger_groups;       /* TaskSwitchingPolicy.prefer_larger_groups  */
  uint8_t proximity_enabled;          /* ProximityOptimizationPolicy.enabled       */
  uint8_t canonical_addresses;        /* 1: every address that enters the mirror goes through pm_address_canonical (what the  */
                                      /* reference's Address parse + to_string does); an id that is not an address is rejected */
                                      /* (discovery entries: skipped, monitor.rs:240,425-429).  0: strings are opaque.        */
} pm_plugin_policy;

typedef struct pm_kv { const char* key; const char* value; } pm_kv;

typedef struct pm_task_desc {         /* shared/src/models/task.rs:162-184 (fields on the path) */
  const char* id;                     /* Uuid as string */
  const char* name;
  const char* image;
  int64_t created_at;
  const pm_kv* env_vars;      uint32_t n_env_vars;      int32_t has_env_vars;      /* Option<HashMap> */
  const char* const* cmd;     uint32_t n_cmd;           int32_t has_cmd;           /* Option<Vec>     */
  const pm_kv* volume_mounts; uint32_t n_volume_mounts; int32_t has_volume_mounts; /* {host_path, container_path} */
  /* scheduling_config (task.rs:58-61): 0 = None; 1 = Some, no "node_groups" plugin entry;
   * 2 = "node_groups" entry without "allowed_topologies"; 3 = allowed_topologies list below */
  int32_t scheduling;
  const char* const* allowed_topologies; uint32_t n_allowed_topologies;
} pm_task_desc;

typedef struct pm_node_desc {         /* orchestrator/src/models/node.rs:10-37 (fields on the path) */
  const char* address;                /* Address::to_string(), opaque, EIP-55 cased by the caller */
  uint32_t status;                    /* NodeStatus ordinal: Discovered=0, WaitingForHeartbeat, Healthy=2,
                                         Unhealthy, Dead=4, Ejected, Banned, LowBalance=7 (node.rs:74-85) */
  const char* p2p_id;                 /* NULL == None */
  uint32_t spec_flags;                /* PM_W_HAS_* presence bits of compute_specs */
  uint32_t gpu_count, gpu_mem_mb;
  const char* gpu_model;
  uint32_t cpu_cores, ram_mb, storage_gb;
  int32_t has_location;
  double lat, lon;
  const char* ip_address;             /* NULL keeps the stored value */
  uint16_t port;
  uint16_t reserved;
  int64_t last_status_change_ms;      /* 0 keeps the stored value (Option<DateTime<Utc>>) */
} pm_node_desc;

typedef struct pm_discovery_node {    /* shared/src/models/node.rs:552-570 (fields the monitor reads) */
  pm_node_desc node;                  /* id (as address), compute_specs, location; status/p2p ignored */
  const char* ip_address;
  uint16_t port;
  uint8_t is_validated, is_active, is_provider_whitelisted, is_blacklisted;
  uint8_t has_latest_balance, latest_balance_is_zero;
  int64_t last_updated_ms;            /* < 0 == None */
} pm_discovery_node;

/* NodeGroupsPlugin::new_with_policy (mod.rs:129-175).  engine may be NULL (then
 * pm_plugin_try_form_new_groups fails with PM_E_NO_DEVICE); policy NULL = defaults. */
int  pm_plugin_create(pm_engine* engine, const pm_plugin_policy* policy, pm_plugin** out);
void pm_plugin_destroy(pm_plugin*);
const char* pm_plugin_last_error(const pm_plugin*);
/* duplicate name / max < min are PM_E_INVALID (the reference panics, mod.rs:141-147);
 * requirements NULL == compute_requirements: None, else ComputeRequirements::from_str */
int pm_plugin_add_config(pm_plugin*, const char* name, uint32_t min_group_size, uint32_t max_group_size,
                         const char* requirements);
int pm_plugin_seal_configs(pm_plugin*);                                   /* the ctor's sort, mod.rs:150-164 */
int pm_plugin_enable_configuration(pm_plugin*, const char* name, int enable);   /* mod.rs:1328-1346 */
int pm_plugin_upsert_node(pm_plugin*, const pm_node_desc*);                /* NodeStore::add_node / update */
int pm_plugin_set_node_status(pm_plugin*, const char* address, uint32_t status); /* + handle_status_change */
/* DiscoveryMonitor: reconcile validated discovery nodes into the table
 * (discovery/monitor.rs:195-435); the Theta(N^2) same-endpoint scan is a hash lookup here. */
int pm_plugin_sync_discovery(pm_plugin*, const pm_discovery_node* nodes, uint32_t n, int64_t now_ms,
                             uint32_t max_healthy_nodes_with_same_endpoint, uint32_t* n_new);
/* same, from the discovery service's wire format: {"success":true,"data":[DiscoveryNode,...]} */
int pm_plugin_sync_discovery_json(pm_plugin*, const char* json, size_t len, int64_t now_ms,
                                  uint32_t max_healthy_nodes_with_same_endpoint, uint32_t* n_new);
int pm_plugin_get_node(pm_plugin*, const char* address, char* buf, size_t len);   /* JSON or null */
int pm_plugin_add_task(pm_plugin*, const pm_task_desc*);                   /* TaskStore::add_task + on_task_created */
int pm_plugin_delete_task(pm_plugin*, const char* id);                     /* delete_task + on_task_deleted */
int pm_plugin_try_form_new_groups(pm_plugin*, uint32_t* n_formed);         /* mod.rs:478-628 via pm_match */
int pm_plugin_try_merge_solo_groups(pm_plugin*, uint32_t* n_merged);       /* mod.rs:631-971 via pm_match */
/* the "upload:<node>:<group>:<file>" key the storage route records; feeds ${TOTAL_UPLOAD_COUNT} */
int pm_plugin_record_upload(pm_plugin*, const char* address, const char* group_id, const char* file_name);
/* JSON out (NUL-terminated into buf): NodeGroup {"id","nodes","configuration_name","task_id"} or null */
int pm_plugin_get_node_group(pm_plugin*, const char* address, char* buf, size_t len);
int pm_plugin_get_all_groups(pm_plugin*, char* buf, size_t len);           /* sorted by id, mod.rs:1040 */
/* get_group_by_id (mod.rs:1046-1055); validate_group_exists (:1067-1070) is `result != null`      */
int pm_plugin_get_group_by_id(pm_plugin*, const char* group_id, char* buf, size_t len);
/* handle_group_not_found (mod.rs:1073-1119): the task of a group that was dissolved under the scheduler goes
 * to the first idle group in get_all_groups() order (SET NX); *reassigned = 1 when one took it      */
int pm_plugin_handle_group_not_found(pm_plugin*, const char* group_id, const char* task_id, uint32_t* reassigned);
/* The node table as the engine's SoA tables (SURVEY 8 A21 / 8f-1), exactly what a management pass uploads: rows in
 * node_store.get_nodes() order (stable status-class sort, node_store.rs:195-206), candidate flags (PM_W_HEALTHY / P2P /
 * ASSIGNED, mod.rs:492-497), locations, BTreeSet<String> address ranks.  Any array may be NULL; capacity in rows.    */
int pm_plugin_export_tables(pm_plugin*, pm_worker_a* a, pm_worker_b* b, double* lat, double* lon, uint32_t* addr_rank,
                            uint32_t capacity, uint32_t* n_rows);
/* The inverse of pm_plugin_redis_writeback, for start-up: a group read back from the reference's keys
 * (`node_group:<id>` JSON + `group_task:<id>`) is put into the tables as it is.  nodes come in the stored
 * (BTreeSet) order; task_id NULL = no claim; created_at_ms < 0 = now.  PM_E_STATE when the id exists or a node is
 * already in a group.  The group id counter moves past ids of the engine's own form (lower-case hex).        */
int pm_plugin_restore_group(pm_plugin*, const char* id, const char* configuration_name, const char* const* nodes,
                            uint32_t n_nodes, const char* task_id, int64_t created_at_ms);
/* Redis write-back in the reference's key formats (mod.rs:25-28,299-322,471-476), as a JSON array of
 * commands, so /groups, /nodes, storage routes and the metrics sync keep working unchanged.        */
int pm_plugin_redis_writeback(pm_plugin*, char* buf, size_t len);
/* Scheduler::get_task_for_node (scheduler/mod.rs:26-74) with the plugin chain
 * [NodeGroupsPlugin] when configurations exist, else [NewestTaskPlugin]:
 * writes {"current_task": Task|null} (shared/src/models/heartbeat.rs:7-22). */
int pm_scheduler_get_task_for_node(pm_plugin*, const char* address, char* buf, size_t len);

#ifdef __cplusplus
}
#endif
#endif /* PRIME_MATCH_H */
