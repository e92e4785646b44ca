// pm_engine.cu — the engine behind include/prime_match.h.
//
// One engine = one CUDA device + one stream.  pm_match() is the management pass
// that replaces NodeGroupsPlugin::try_form_new_groups (reference
// crates/orchestrator/src/plugins/node_groups/mod.rs:478-628): for tiles of asks
// (configurations, priority order) x all candidate workers it builds the int64
// cost matrix in HBM, reduces it (per-ask argmin, per-worker first feasible ask)
// and then runs the resolution sweep that reproduces the reference's sequential
// greedy allocation bit for bit.  There is no CPU fallback: without an sm_100
// device pm_create fails with PM_E_NO_DEVICE.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <dlfcn.h>
#include <nccl.h>   // types and prototypes only: the library is resolved at run time (nccl_api below), never linked

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "pm_guard.hpp"
#include "pm_kernels.cuh"
#include "pm_proximity.cuh"
#include "pm_proximity_band.cuh"
#include "pm_proximity_grid.cuh"
#include "pm_auction.cuh"

struct pm_engine;

namespace {

std::string g_create_error;

template <class T> struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  cudaError_t ensure(size_t want) {
    if (want <= n && p) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
    if (want == 0) want = 1;
    cudaError_t e = cudaMalloc(&p, want * sizeof(T));
    if (e == cudaSuccess) n = want;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
  // capacity >= want, the first `keep` elements preserved, everything after them zero
  cudaError_t grow_keep(size_t want, size_t keep, cudaStream_t st) {
    if (want <= n && p) return cudaSuccess;
    const size_t cap = std::max<size_t>(want + want / 4, 1);
    T* q = nullptr;
    cudaError_t e = cudaMalloc(&q, cap * sizeof(T));
    if (e != cudaSuccess) return e;
    keep = p ? std::min(keep, n) : 0;
    if (keep) e = cudaMemcpyAsync(q, p, keep * sizeof(T), cudaMemcpyDeviceToDevice, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(q + keep, 0, (cap - keep) * sizeof(T), st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { cudaFree(q); return e; }
    if (p) cudaFree(p);
    p = q;
    n = cap;
    return cudaSuccess;
  }
};
template <class T> struct PinBuf {
  T* p = nullptr;
  size_t n = 0;
  cudaError_t ensure(size_t want) {
    if (want <= n && p) return cudaSuccess;
    if (p) cudaFreeHost(p);
    p = nullptr;
    n = 0;
    if (want == 0) want = 1;
    cudaError_t e = cudaMallocHost(&p, want * sizeof(T));
    if (e == cudaSuccess) n = want;
    return e;
  }
  void release() {
    if (p) cudaFreeHost(p);
    p = nullptr;
    n = 0;
  }
};

inline unsigned blocks_for(size_t n, unsigned threads) { return (unsigned)((n + threads - 1) / threads); }

// NCCL is plumbing for the one exchange of a sharded pass.  It is looked up at run time so that the library loads
// (and every single-GPU path works) on hosts without it: first among the symbols already in the process (a host that
// has NCCL loaded, e.g. through torch, shares its copy), then by soname.
struct NcclApi {
  decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
  decltype(&ncclCommInitRank) CommInitRank = nullptr;
  decltype(&ncclCommInitAll) CommInitAll = nullptr;
  decltype(&ncclCommDestroy) CommDestroy = nullptr;
  decltype(&ncclCommAbort) CommAbort = nullptr;
  decltype(&ncclAllGather) AllGather = nullptr;
  decltype(&ncclGetErrorString) GetErrorString = nullptr;
  bool ok = false;
  std::string err;
};
const NcclApi& nccl_api() {
  static const NcclApi api = [] {
    NcclApi a;
    void* h = dlsym(RTLD_DEFAULT, "ncclAllGather") ? RTLD_DEFAULT : nullptr;
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) { a.err = "NCCL not found (libnccl.so.2): multi-GPU matching needs it"; return a; }
#define PM_NCCL_SYM(name) a.name = reinterpret_cast<decltype(a.name)>(dlsym(h, "nccl" #name)); if (!a.name) { a.err = "libnccl: missing nccl" #name; return a; }
    PM_NCCL_SYM(GetUniqueId) PM_NCCL_SYM(CommInitRank) PM_NCCL_SYM(CommInitAll) PM_NCCL_SYM(CommDestroy)
    PM_NCCL_SYM(CommAbort) PM_NCCL_SYM(AllGather) PM_NCCL_SYM(GetErrorString)
#undef PM_NCCL_SYM
    a.ok = true;
    return a;
  }();
  return api;
}

}  // namespace

struct pm_comm {
  ncclComm_t nccl = nullptr;
  uint32_t n_ranks = 1, rank = 0;
  int device = 0;
};

struct pm_engine {
  pm_cfg cfg{};
  int device = 0;
  cudaStream_t stream = nullptr;
  std::string err;
  std::mutex mu;

  // tables
  uint32_t n_workers = 0, n_asks = 0, n_opts = 0;
  uint32_t n_patterns = 0, n_models = 0, words = 1;
  uint32_t max_pattern_row = 0;
  bool have_workers = false, have_asks = false, have_bits = false, have_loc = false, have_rank = false;
  bool all_solo = true;  // every ask has min == max == 1
  int tune_cost = 0;   // PM_TUNE_COST=8: the int64 cost tile even where 16-bit price words would do (in-binary A/B)
  int tune_argmin = 0, tune_generic = 0, tune_build = 0, tune_auction = 0, tune_prox = 0, tune_auc_good = 0, tune_auc_extra = 0;   // PM_TUNE_ARGMIN: kernel-shape experiments (see profiles/)
  DevBuf<uint4> wa, wb;
  DevBuf<double> lat, lon;
  DevBuf<uint32_t> addr_rank;
  DevBuf<pm::DevAsk> asks;
  DevBuf<pm::DevOpt> opts;
  DevBuf<pm::DevOptF> opts_fast;
  DevBuf<pm::FastRow> frows;
  bool rows_bound = false;     // FastRow.wp matches the current model table (pm_bind_rows)
  bool rows_bound_wm = false;  // ... bound to the worker-major one-word table
  DevBuf<uint32_t> nacc, bits_wm;   // worker-major acceptance (pm_worker_nacc) and its one-word table ~(1 << row)
  bool nacc_valid = false;
  DevBuf<pm_ask> raw_asks;
  DevBuf<pm_gpu_opt> raw_opts;
  DevBuf<uint32_t> ask_counts, ask_newoff;
  bool asks_small = true;      // every ask operand fits the fast predicate (pm_device.cuh DevOptF)
  bool workers_small = false;  // ... and every worker operand (checked on the device)
  bool workers_checked = false;
  bool prices_narrow = false;  // every ext_ask_price <= 0xFFFE: the cost tile can hold 16-bit price words (same check)
  DevBuf<uint32_t> amin, amax, bits;
  DevBuf<uint32_t> scratch_idx, scratch_flags;
  DevBuf<uint4> upd_a, upd_b;          // staging of pm_update_workers
  DevBuf<double> upd_lat, upd_lon;
  uint64_t table_version = 0;          // bumped by every call that changes a table (pm_table_version)

  // evaluation
  DevBuf<unsigned char> cost;   // the materialised cost tile (int64 keys or 16-bit price words), sized in bytes
  DevBuf<uint32_t> first_ask, ask_count;
  DevBuf<long long> ask_best;

  // resolution
  DevBuf<uint32_t> keys, keys_sorted, iota, order, hist, seg_start, ngroups, group_base;
  DevBuf<uint32_t> base_len, xhead, xnext, xcount, popped, counters;  // counters: [0]=any_bad [1]=n_bumped
  DevBuf<unsigned char> cub_tmp;
  DevBuf<uint32_t> prox_list, prox_xs, members_raw;
  DevBuf<double> prox_dist, prox_lat_key;
  DevBuf<uint32_t> prox_lat_ord, prox_rank_of;
  DevBuf<double> pg_part_d, pg_clat, pg_clon, pg_ccos;
  DevBuf<uint32_t> pg_part_i, pg_cta_cnt, pg_ctl;
  int coop_blocks = -1;   // co-resident CTAs of pm_proximity_grid on this device (0: cooperative launch unavailable)
  bool any_max_zero = false;
  // extension (auction) state
  DevBuf<uint32_t> price_cap, auc_owner, auc_assigned, auc_withdrawn, auc_active, auc_bid_w, auc_winner, auc_flag, auc_gidx;
  DevBuf<long long> auc_price, auc_bid_p, auc_bid_max, auc_theta;
  DevBuf<uint32_t> auc_cand, auc_theta_w, auc_pool, auc_pool_bound_w;
  DevBuf<long long> auc_pool_bound_v;
  DevBuf<uint32_t> auc_class_of, auc_class_rep, auc_class_req, auc_class_list, auc_retry, auc_fallback;
  DevBuf<uint32_t> auc_walk_list, auc_split_w, auc_split_ticket;
  DevBuf<long long> auc_split_v;
  DevBuf<uint32_t> auc_perm, auc_pos_of, auc_idx, auc_sorted, auc_incl;
  DevBuf<uint64_t> auc_hash, auc_hash_out, auc_ckey, auc_ckey_s;
  DevBuf<uint4> auc_wa_s, auc_wb_s;
  DevBuf<long long> auc_price_s;
  DevBuf<pm::AuctionCtl> auc_ctl;
  PinBuf<pm::AuctionCtl> h_ctl;
  uint32_t auc_n_classes = 0;
  bool auc_classes_valid = false;
  bool have_caps = false;
  DevBuf<uint32_t> auc_split_first;
  DevBuf<uint64_t> auc_skip_key;
  DevBuf<uint32_t> reputation, ask_min_rep, auc_rep_s;   // extension: worker reputation column, per-ask floor, sorted copy
  bool have_rep = false, have_min_rep = false;
  uint64_t auc_scale = 1, auc_eps_start = 1;
  uint32_t auc_eps_div = 4;
  DevBuf<uint32_t> worker_group, worker_ask, group_ask, group_off, members;
  PinBuf<uint32_t> h_scalars;  // small D2H mailbox

  // result (pinned host)
  PinBuf<uint32_t> r_worker_group, r_worker_ask, r_group_ask, r_group_off, r_members, r_ask_count;
  PinBuf<long long> r_ask_best;
  uint32_t n_groups = 0, n_assigned = 0;
  bool matched = false, local_done = false;

  // multi-GPU: the communicator this engine exchanges through (not owned), and the packed exchange buffers
  pm_comm* comm = nullptr;
  DevBuf<unsigned char> xchg_send, xchg_recv;

  // The contiguous canonical-order range of workers this engine evaluates: the whole table, the range fixed by
  // pm_cfg / pm_set_shard, or — with a communicator attached — the rank's equal share.
  void shard(uint32_t* w0, uint32_t* nw) const {
    const uint32_t W = n_workers;
    if (comm) {
      const uint32_t per = (uint32_t)(((uint64_t)W + comm->n_ranks - 1) / comm->n_ranks);
      *w0 = (uint32_t)std::min<uint64_t>((uint64_t)comm->rank * per, W);
      *nw = std::min(per, W - *w0);
    } else {
      *w0 = cfg.shard_first;
      *nw = cfg.shard_count ? cfg.shard_count : (W > *w0 ? W - *w0 : 0);
    }
  }

  pm_stats stats{};
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  bool own_stream = true;
  struct TimedRegion { cudaEvent_t a, b; float* acc; };
  std::vector<cudaEvent_t> ev_pool;     // grows on demand, reused across matches
  std::vector<TimedRegion> ev_pending;
  size_t ev_used = 0;
  cudaEvent_t take_event() {
    if (ev_used == ev_pool.size()) {
      cudaEvent_t ev = nullptr;
      if (cudaEventCreate(&ev) != cudaSuccess) return nullptr;
      ev_pool.push_back(ev);
    }
    return ev_pool[ev_used++];
  }
  void resolve_timers() {  // caller has synchronised the stream
    for (auto& r : ev_pending) {
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) *r.acc += ms;
    }
    ev_pending.clear();
    ev_used = 0;
  }

  int fail(pm_status st, const std::string& msg) {
    err = msg;
    return st;
  }
};

#define PM_CUDA(call)                                                                   \
  do {                                                                                  \
    cudaError_t _e = (call);                                                            \
    if (_e != cudaSuccess) {                                                            \
      return e->fail(PM_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(_e));    \
    }                                                                                   \
  } while (0)

#define PM_LAUNCH_CHECK(name)                                                           \
  do {                                                                                  \
    cudaError_t _e = cudaGetLastError();                                                \
    if (_e != cudaSuccess)                                                              \
      return e->fail(PM_E_CUDA, std::string("launch ") + name + ": " + cudaGetErrorString(_e)); \
    ++e->stats.n_launches;                                                              \
  } while (0)

namespace {

// Per-launch CUDA-event timing without host synchronisation: start/stop events
// are recorded on the engine stream around a region and resolved in one go at
// the end of the match (which synchronises anyway to read the group count).
struct Timer {
  pm_engine* e;
  float* acc;
  bool on;
  size_t slot = 0;
  Timer(pm_engine* e_, float* acc_);
  void stop();
};

Timer::Timer(pm_engine* e_, float* acc_) : e(e_), acc(acc_), on((e_->cfg.flags & PM_CFG_TIMING) != 0) {
  if (!on) return;
  cudaEvent_t a = e->take_event(), b = e->take_event();
  if (!a || !b) { on = false; return; }
  slot = e->ev_pending.size();
  e->ev_pending.push_back({a, b, acc});
  cudaEventRecord(a, e->stream);
}
void Timer::stop() {
  if (!on) return;
  cudaEventRecord(e->ev_pending[slot].b, e->stream);
  on = false;
}

pm::EvalParams eval_params(pm_engine* e) {
  pm::EvalParams p;
  p.wa = e->wa.p;
  p.wb = e->wb.p;
  p.asks = e->asks.p;
  p.opts = e->opts.p;
  p.opts_fast = e->opts_fast.p;
  p.frows = e->frows.p;
  p.bits = e->bits.p;
  p.nacc = nullptr;
  p.words = e->words;
  p.n_workers = e->n_workers;
  p.n_asks = e->n_asks;
  p.n_opts = e->n_opts;
  p.n_bits_rows = e->have_bits ? e->n_patterns + 1 : 1;
  p.sign_shift = 31;
  return p;
}

}  // namespace

extern "C" {

void* pm_alloc_pinned(size_t bytes) {
  void* p = nullptr;
  if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return p;
}
void pm_free_pinned(void* p) {
  if (p) cudaFreeHost(p);
}

int pm_create(const pm_cfg* cfg, pm_engine** out) try {
  if (!cfg || !out) {
    g_create_error = "pm_create: null argument";
    return PM_E_INVALID;
  }
  *out = nullptr;
  if (cfg->abi_version != PM_ABI_VERSION) {
    g_create_error = "pm_create: ABI version mismatch";
    return PM_E_INVALID;
  }
  int ndev = 0;
  cudaError_t ce = cudaGetDeviceCount(&ndev);
  if (ce != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    g_create_error = "pm_create: no CUDA device visible (this engine has no CPU path)";
    return PM_E_NO_DEVICE;
  }
  if (cfg->device < 0 || cfg->device >= ndev) {
    g_create_error = "pm_create: device ordinal out of range";
    return PM_E_INVALID;
  }
  cudaDeviceProp prop{};
  if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess || prop.major < 10) {
    cudaGetLastError();
    g_create_error = "pm_create: device is not sm_100 or newer (kernels are built for sm_100a only)";
    return PM_E_NO_DEVICE;
  }
  pm_engine* e = new (std::nothrow) pm_engine;
  if (!e) return PM_E_NOMEM;
  e->cfg = *cfg;
  if (e->cfg.cost_tile_bytes == 0) e->cfg.cost_tile_bytes = 8ull << 30;
  e->device = cfg->device;
  if (const char* t = std::getenv("PM_TUNE_ARGMIN")) e->tune_argmin = std::atoi(t);
  if (const char* t = std::getenv("PM_TUNE_GENERIC")) e->tune_generic = std::atoi(t);
  if (const char* t = std::getenv("PM_TUNE_BUILD")) e->tune_build = std::atoi(t);
  if (const char* t = std::getenv("PM_TUNE_COST")) e->tune_cost = std::atoi(t);
  if (const char* t = std::getenv("PM_TUNE_AUCTION")) e->tune_auction = std::atoi(t);
  if (const char* t = std::getenv("PM_TUNE_AUCTION_POOL")) std::sscanf(t, "%d,%d", &e->tune_auc_good, &e->tune_auc_extra);   // pool fill of a class walk
  if (const char* t = std::getenv("PM_TUNE_PROX")) e->tune_prox = std::atoi(t);   // 0: all-SM cooperative sweep; 2: single-CTA sweep; 1: latitude-banded single-CTA sweep (experimental)
  bool ok = cudaSetDevice(e->device) == cudaSuccess;
  if (ok && cfg->stream) {
    e->stream = (cudaStream_t)cfg->stream;  // caller's stream (e.g. torch's current stream)
    e->own_stream = false;
  } else if (ok) {
    ok = cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) == cudaSuccess;
  }
  ok = ok &&
            cudaEventCreate(&e->ev0) == cudaSuccess && cudaEventCreate(&e->ev1) == cudaSuccess &&
            e->h_scalars.ensure(64) == cudaSuccess && e->counters.ensure(32) == cudaSuccess;
  if (!ok) {
    g_create_error = std::string("pm_create: ") + cudaGetErrorString(cudaGetLastError());
    delete e;
    return PM_E_CUDA;
  }
  *out = e;
  return PM_OK;
} catch (...) { return pm_guard_rc(); }

void pm_destroy(pm_engine* e) {
  if (!e) return;
  cudaSetDevice(e->device);
  if (e->stream) cudaStreamSynchronize(e->stream);
  e->wa.release(); e->wb.release(); e->lat.release(); e->lon.release(); e->addr_rank.release();
  e->asks.release(); e->opts.release(); e->opts_fast.release(); e->frows.release();
  e->raw_asks.release(); e->raw_opts.release(); e->ask_counts.release(); e->ask_newoff.release(); e->amin.release(); e->amax.release(); e->bits.release();
  e->scratch_idx.release(); e->scratch_flags.release();
  e->upd_a.release(); e->upd_b.release(); e->upd_lat.release(); e->upd_lon.release();
  e->cost.release(); e->first_ask.release(); e->ask_count.release(); e->ask_best.release();
  e->keys.release(); e->keys_sorted.release(); e->iota.release(); e->order.release();
  e->hist.release(); e->seg_start.release(); e->ngroups.release(); e->group_base.release();
  e->base_len.release(); e->xhead.release(); e->xnext.release(); e->xcount.release();
  e->popped.release(); e->counters.release(); e->cub_tmp.release();
  e->prox_list.release(); e->prox_xs.release(); e->members_raw.release(); e->prox_dist.release();
  e->prox_lat_key.release(); e->prox_lat_ord.release(); e->prox_rank_of.release();
  e->pg_part_d.release(); e->pg_part_i.release(); e->pg_cta_cnt.release(); e->pg_ctl.release();
  e->pg_clat.release(); e->pg_clon.release(); e->pg_ccos.release();
  e->nacc.release(); e->bits_wm.release();
  e->reputation.release(); e->ask_min_rep.release(); e->auc_rep_s.release(); e->auc_split_first.release(); e->auc_skip_key.release();
  e->price_cap.release(); e->auc_owner.release(); e->auc_assigned.release(); e->auc_withdrawn.release();
  e->auc_active.release(); e->auc_bid_w.release(); e->auc_winner.release(); e->auc_flag.release(); e->auc_gidx.release();
  e->auc_price.release(); e->auc_bid_p.release(); e->auc_bid_max.release();
  e->auc_theta.release(); e->auc_cand.release(); e->auc_theta_w.release();
  e->auc_walk_list.release(); e->auc_split_w.release(); e->auc_split_ticket.release(); e->auc_split_v.release();
  e->auc_pool.release(); e->auc_pool_bound_w.release(); e->auc_pool_bound_v.release(); e->auc_ckey.release(); e->auc_ckey_s.release();
  e->auc_class_of.release(); e->auc_class_rep.release(); e->auc_class_req.release(); e->auc_class_list.release();
  e->auc_retry.release(); e->auc_fallback.release(); e->auc_perm.release(); e->auc_pos_of.release();
  e->auc_idx.release(); e->auc_sorted.release(); e->auc_incl.release(); e->auc_hash.release();
  e->auc_hash_out.release(); e->auc_wa_s.release(); e->auc_wb_s.release(); e->auc_price_s.release(); e->auc_ctl.release();
  e->h_ctl.release();
  e->worker_group.release(); e->worker_ask.release(); e->group_ask.release();
  e->group_off.release(); e->members.release(); e->h_scalars.release();
  e->xchg_send.release(); e->xchg_recv.release();
  e->r_worker_group.release(); e->r_worker_ask.release(); e->r_group_ask.release();
  e->r_group_off.release(); e->r_members.release(); e->r_ask_count.release(); e->r_ask_best.release();
  if (e->ev0) cudaEventDestroy(e->ev0);
  if (e->ev1) cudaEventDestroy(e->ev1);
  for (cudaEvent_t ev : e->ev_pool) cudaEventDestroy(ev);
  if (e->stream && e->own_stream) cudaStreamDestroy(e->stream);
  delete e;
}

const char* pm_last_error(const pm_engine* e) { return e ? e->err.c_str() : g_create_error.c_str(); }

int pm_set_asks(pm_engine* e, const pm_ask* asks, uint32_t n_asks, const pm_gpu_opt* opts,
                uint32_t n_opts) try {
  if (!e) return PM_E_INVALID;
  std::lock_guard<std::mutex> lk(e->mu);
  ++e->table_version;
  if ((n_asks && !asks) || (n_opts && !opts)) return e->fail(PM_E_INVALID, "pm_set_asks: null table");
  if (n_asks >= (1u << 30)) return e->fail(PM_E_INVALID, "pm_set_asks: too many asks");
  PM_CUDA(cudaSetDevice(e->device));
  // the caller's tables go up as they are; the device converts them (pm_ask_convert)
  PM_CUDA(e->raw_asks.ensure(n_asks)); PM_CUDA(e->raw_opts.ensure(n_opts));
  PM_CUDA(e->ask_counts.ensure((size_t)n_asks + 1)); PM_CUDA(e->ask_newoff.ensure((size_t)n_asks + 1));
  PM_CUDA(e->asks.ensure(n_asks)); PM_CUDA(e->amin.ensure(n_asks)); PM_CUDA(e->amax.ensure(n_asks));
  // asks may share or overlap option rows, so the converted table (one private range per ask) can be longer than
  // the caller's: size it by the sum of the per-ask counts
  uint64_t opt_rows = 0;
  for (uint32_t i = 0; i < n_asks; ++i) opt_rows += std::max<uint32_t>(asks[i].n_opts, 1u);   // an ask without options gets a neutral row
  if (opt_rows >= (1ull << 31)) return e->fail(PM_E_INVALID, "pm_set_asks: too many option rows");
  const size_t opt_cap = std::max<size_t>(n_opts, (size_t)opt_rows);
  PM_CUDA(e->opts.ensure(opt_cap)); PM_CUDA(e->opts_fast.ensure(opt_cap)); PM_CUDA(e->frows.ensure(n_asks));
  e->rows_bound = false;
  if (n_asks) PM_CUDA(cudaMemcpyAsync(e->raw_asks.p, asks, (size_t)n_asks * sizeof(pm_ask), cudaMemcpyHostToDevice, e->stream));
  if (n_opts) PM_CUDA(cudaMemcpyAsync(e->raw_opts.p, opts, (size_t)n_opts * sizeof(pm_gpu_opt), cudaMemcpyHostToDevice, e->stream));
  PM_CUDA(cudaMemsetAsync(e->counters.p + 12, 0, 8, e->stream));
  pm::pm_ask_counts<<<blocks_for((size_t)n_asks + 1, 256), 256, 0, e->stream>>>(e->raw_asks.p, n_asks, n_opts, e->ask_counts.p, e->counters.p + 12);
  PM_LAUNCH_CHECK("pm_ask_counts");
  {
    size_t tmp = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp, e->ask_counts.p, e->ask_newoff.p, (int)(n_asks + 1), e->stream);
    PM_CUDA(e->cub_tmp.ensure(tmp));
    PM_CUDA(cub::DeviceScan::ExclusiveSum(e->cub_tmp.p, tmp, e->ask_counts.p, e->ask_newoff.p, (int)(n_asks + 1), e->stream));
  }
  if (n_asks) {
    pm::pm_ask_convert<<<blocks_for(n_asks, 256), 256, 0, e->stream>>>(e->raw_asks.p, e->raw_opts.p, n_asks, e->ask_newoff.p, e->asks.p,
                                                                        e->opts.p, e->opts_fast.p, e->amin.p, e->amax.p,
                                                                        e->counters.p + 12, e->counters.p + 13, e->frows.p);
    PM_LAUNCH_CHECK("pm_ask_convert");
  }
  PM_CUDA(cudaMemcpyAsync(e->h_scalars.p + 20, e->counters.p + 12, 8, cudaMemcpyDeviceToHost, e->stream));
  PM_CUDA(cudaMemcpyAsync(e->h_scalars.p + 22, e->ask_newoff.p + n_asks, 4, cudaMemcpyDeviceToHost, e->stream));
  PM_CUDA(cudaStreamSynchronize(e->stream));  // also: the caller's tables are no longer read after return
  const uint32_t st = e->h_scalars.p[20];
  e->have_asks = false;
  // NodeGroupConfiguration::is_valid, mod.rs:55-60 (the reference panics at construction)
  if (st & pm::kAskBadSizes)
    return e->fail(PM_E_INVALID, "pm_set_asks: max_group_size < min_group_size (Plugin configuration is invalid)");
  if (st & pm::kAskBadRange) return e->fail(PM_E_INVALID, "pm_set_asks: option range out of bounds");
  e->n_asks = n_asks;
  e->n_opts = e->h_scalars.p[22];
  e->max_pattern_row = e->h_scalars.p[21];
  e->all_solo = (st & pm::kAskNotSolo) == 0;
  e->asks_small = (st & pm::kAskNotSmall) == 0;
  e->any_max_zero = (st & pm::kAskMaxZero) != 0;
  e->have_caps = false;
  e->have_min_rep = false;
  e->auc_classes_valid = false;
  e->have_asks = true;
  e->matched = e->local_done = false;
  return PM_OK;
} catch (...) { return pm_guard_rc(); }

int pm_set_model_table(pm_engine* e, const uint32_t* bits, uint32_t n_patterns, uint32_t n_models,
                       uint32_t words) try {
  if (!e) return PM_E_INVALID;
  std::lock_guard<std::mutex> lk(e->mu);
  ++e->table_version;
  if (words == 0) words = 1;
  if (n_patterns && !bits) return e->fail(PM_E_INVALID, "pm_set_model_table: null table");
  if ((uint64_t)words * 32 < n_models) return e->fail(PM_E_INVALID, "pm_set_model_table: words too small");
  // device layout: 31 models per word (bit 31 stays clear: the fast predicate turns "non-zero" into a sign bit by
  // an addition, pm_device.cuh DevOptF), row 0 = no model clause = accepts everything
  const uint32_t dwords = std::max<uint32_t>((n_models + pm::kModelsPerWord - 1) / pm::kModelsPerWord, 1u);
  std::vector<uint32_t> tbl((size_t)(n_patterns + 1) * dwords, 0u);
  for (uint32_t i = 0; i < dwords; ++i) tbl[i] = 0x7FFFFFFFu;
  for (uint32_t p = 0; p < n_patterns; ++p) {
    const uint32_t* src = bits + (size_t)p * words;
    uint32_t* dst = tbl.data() + (size_t)(p + 1) * dwords;
    for (uint32_t wi = 0; wi < words; ++wi) {
      uint32_t v = src[wi];
      while (v) {
        const uint32_t m = wi * 32u + (uint32_t)__builtin_ctz(v);
        v &= v - 1;
        if (m < n_models) dst[m / pm::kModelsPerWord] |= 1u << (m % pm::kModelsPerWord);
      }
    }
  }
  words = dwords;
  PM_CUDA(cudaSetDevice(e->device));
  PM_CUDA(e->bits.ensure(tbl.size()));
  PM_CUDA(cudaMemcpyAsync(e->bits.p, tbl.data(), tbl.size() * 4, cudaMemcpyHostToDevice, e->stream));
  PM_CUDA(cudaStreamSynchronize(e->stream));
  e->n_patterns = n_patterns;
  e->n_models = n_models;
  e->words = words;
  e->have_bits = true;
  e->rows_bound = false;
  e->nacc_valid = false;
  e->matched = e->local_done = false;
  return PM_OK;
} catch (...) { return pm_guard_rc(); }

int pm_set_worker_count(pm_engine* e, uint32_t n_workers) try {
  if (!e) return PM_E_INVALID;
  std::lock_guard<std::mutex> lk(e->mu);
  ++e->table_version;
  PM_CUDA(cudaSetDevice(e->device));
  if (n_workers > e->wa.n || !e->wa.p) {
    // grow, preserving nothing: callers upsert after (re)sizing
    PM_CUDA(e->wa.ensure(n_workers));
    PM_CUDA(e->wb.ensure(n_workers));
  }
  PM_CUDA(cudaMemsetAsync(e->wa.p, 0, (size_t)std::max<uint32_t>(n_workers, 1) * 16, e->stream));
  PM_CUDA(cudaMemsetAsync(e->wb.p, 0, (size_t)std::max<uint32_t>(n_workers, 1) * 16, e->stream));
  e->n_workers = n_workers;
  e->workers_checked = false;
  e->nacc_valid = false;
  e->have_workers = true;
  e->have_loc = e->have_rank = false;
  e->have_rep = false;
  e->matched = e->local_done = false;
  return PM_OK;
} catch (...) { return pm_guard_rc(); }

int pm_upsert_workers(pm_engine* e, const pm_worker_a* a, const pm_worker_b* b, uint32_t first,
                      uint32_t n) try {
  if (!e) return PM_E_INVALID;
  std::lock_guard<std::mutex> lk(e->mu);
  ++e->table_version;
  if (!e->have_workers) return e->fail(PM_E_STATE, "pm_upsert_workers: call pm_set_worker_count first");
  if ((uint64_t)first + n > e->n_workers) return e->fail(PM_E_INVALID, "pm_upsert_workers: range out of bounds");
  if (n && (!a || !b)) return e->fail(PM_E_INVALID, "pm_upsert_workers: null plane");
  PM_CUDA(cudaSetDevice(e->device));
  if (n) {
    PM_CUDA(cudaMemcpyAsync(e->wa.p + first, a, (size_t)n * 16, cudaMemcpyHostToDevice, e->stream));
    PM_CUDA(cudaMemcpyAsync(e->wb.p + first, b, (size_t)n * 16, cudaMemcpyHostToDevice, e->stream));
  }
  e->workers_checked = false;
  e->nacc_valid = false;
  e->matched = e->local_done = false;
  return PM_OK;
} catch (...) { return pm_guard_rc(); }

int pm_set_worker_locations(pm_engine* e, const double* lat, const double* lon, uint32_t first,
                            uint32_t n) try {
  if (!e) return PM_E_INVALID;
  std::lock_guard<std::mutex> lk(e->mu);
  ++e->table_version;
  if (!e->have_workers) return e->fail(PM_E_STATE, "pm_set_worker_locations: no worker table");
  if ((uint64_t)first + n > e->n_workers) return e->fail(PM_E_INVALID, "pm_set_worker_locations: range");
  PM_CUDA(cudaSetDevice(e->device));
  PM_CUDA(e->lat.ensure(e->n_workers));
  PM_CUDA(e->lon.ensure(e->n_workers));
  if (n) {
    PM_CUDA(cudaMemcpyAsync(e->lat.p + first, lat, (size_t)n * 8, cudaMemcpyHostToDevice, e->stream));
    PM_CUDA(cudaMemcpyAsync(e->lon.p + first, lon, (size_t)n * 8, cudaMemcpyHostToDevice, e->stream));
  }
  e->have_loc = true;
  return PM_OK;
} catch (...) { return pm_guard_rc(); }

int pm_set_worker_addr_rank(pm_engine* e, const uint32_t* rank, uint32_t first, uint32_t n) try {
  if (!e) return PM_E_INVALID;
  std::lock_guard<std::mutex> lk(e->mu);
  ++e->table_version;
  if (!e->have_workers) return e->fail(PM_E_STATE, "pm_set_worker_addr_rank: no worker table");
  if ((uint64_t)first + n > e->n_workers) return e->fail(PM_E_INVALID, "pm_set_worker_addr_rank: range");
  PM_CUDA(cudaSetDevice(e->device));
  PM_CUDA(e->addr_rank.ensure(e->n_workers));
  if (n) PM_CUDA(cudaMemcpyAsync(e->addr_rank.p + first, rank, (size_t)n * 4, cudaMemcpyHostToDevice, e->stream));
  e->have_rank = true;
  return PM_OK;
} catch (...) { return pm_guard_rc(); }

int pm_set_flags(pm_engine* e, const uint32_t* idx, const uint32_t* flags, uint32_t n) try {
  if (!e) return PM_E_INVALID;
  std::lock_guard<std::mutex> lk(e->mu);
  ++e->table_version;
  if (!e->have_workers) return e->fail(PM_E_STATE, "pm_set_flags: no worker table");
  if (n == 0) return PM_OK;
  if (!idx || !flags) return e->fail(PM_E_INVALID, "pm_set_flags: null");
  PM_CUDA(cudaSetDevice(e->device));
  PM_CUDA(e->scratch_idx.ensure(n));
  PM_CUDA(e->scratch_flags.ensure(n));
  PM_CUDA(cudaMemcpyAsync(e->scratch_idx.p, idx, (size_t)n * 4, cudaMemcpyHostToDevice, e->stream));
  PM_CUDA(cudaMemcpyAsync(e->scratch_flags.p, flags, (size_t)n * 4, cudaMemcpyHostToDevice, e->stream));
  pm::pm_scatter_flags<<<blocks_for(n, 256), 256, 0, e->stream>>>(e->wa.p, e->scratch_idx.p, e->scratch_flags.p, n, e->n_workers);
  PM_LAUNCH_CHECK("pm_scatter_flags");
  e->workers_checked = false;
  e->nacc_valid = false;
  e->matched = e->local_done = false;
  return PM_OK;
} catch (...) { return pm_guard_rc(); }

// Resident tables with deltas (the management pass of a long-running host: only rows that changed travel).
int pm_resize_workers(pm_engine* e, uint32_t n_workers) try {
  if (!e) return PM_E_INVALID;
  std::lock_guard<std::mutex> lk(e->mu);
  ++e->table_version;
  PM_CUDA(cudaSetDevice(e->device));
  const size_t keep = e->have_workers ? e->n_workers : 0;
  PM_CUDA(e->wa.grow_keep(std::max<uint32_t>(n_workers, 1), keep, e->stream));
  PM_CUDA(e->wb.grow_keep(std::max<uint32_t>(n_workers, 1), keep, e->stream));
  if (e->have_loc) {
    PM_CUDA(e->lat.grow_keep(std::max<uint32_t>(n_workers, 1), keep, e->stream));
    PM_CUDA(e->lon.grow_keep(std::max<uint32_t>(n_workers, 1), keep, e->stream));
  }
  if (e->have_rank) PM_CUDA(e->addr_rank.grow_keep(std::max<uint32_t>(n_workers, 1), keep, e->stream));
  if (e->have_rep) PM_CUDA(e->reputation.grow_keep(std::max<uint32_t>(n_workers, 1), keep, e->stream));
  if (n_workers > keep) {   // rows that were beyond the old table (or were cut off earlier) start empty
    PM_CUDA(cudaMemsetAsync(e->wa.p + keep, 0, (size_t)(n_workers - keep) * 16, e->stream));
    PM_CUDA(cudaMemsetAsync(e->wb.p + keep, 0, (size_t)(n_workers - keep) * 16, e->stream));
    if (e->have_loc) {
      PM_CUDA(cudaMemsetAsync(e->lat.p + keep, 0, (size_t)(n_workers - keep) * 8, e->stream));
      PM_CUDA(cudaMemsetAsync(e->lon.p + keep, 0, (size_t)(n_workers - keep) * 8, e->stream));
    }
    if (e->have_rank) PM_CUDA(cudaMemsetAsync(e->addr_rank.p + keep, 0, (size_t)(n_workers - keep) * 4, e->stream));
    if (e->have_rep) PM_CUDA(cudaMemsetAsync(e->reputation.p + keep, 0, (size_t)(n_workers - keep) * 4, e->stream));
  }
  e->n_workers = n_workers;
  e->have_workers = true;
  e->workers_checked = false;
  e->nacc_valid = false;
  e->matched = e->local_done = false;
  return PM_OK;
} catch (...) { return pm_guard_rc(); }

int pm_update_workers(pm_engine* e, const uint32_t* idx, const pm_worker_a* a, const pm_worker_b* b, const double* lat,
                      const double* lon, uint32_t n) try {
  if (!e) return PM_E_INVALID;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->have_workers) return e->fail(PM_E_STATE, "pm_update_workers: no worker table");
  if (n == 0) return PM_OK;
  if (!idx || !a || !b || ((lat == nullptr) != (lon == nullptr))) return e->fail(PM_E_INVALID, "pm_update_workers: null");
  ++e->table_version;
  PM_CUDA(cudaSetDevice(e->device));
  PM_CUDA(e->scratch_idx.ensure(n)); PM_CUDA(e->upd_a.ensure(n)); PM_CUDA(e->upd_b.ensure(n));
  PM_CUDA(cudaMemcpyAsync(e->scratch_idx.p, idx, (size_t)n * 4, cudaMemcpyHostToDevice, e->stream));
  PM_CUDA(cudaMemcpyAsync(e->upd_a.p, a, (size_t)n * 16, cudaMemcpyHostToDevice, e->stream));
  PM_CUDA(cudaMemcpyAsync(e->upd_b.p, b, (size_t)n * 16, cudaMemcpyHostToDevice, e->stream));
  if (lat) {
    if (!e->have_loc) {
      PM_CUDA(e->lat.ensure(e->wa.n)); PM_CUDA(e->lon.ensure(e->wa.n));
      PM_CUDA(cudaMemsetAsync(e->lat.p, 0, e->wa.n * 8, e->stream));
      PM_CUDA(cudaMemsetAsync(e->lon.p, 0, e->wa.n * 8, e->stream));
      e->have_loc = true;
    }
    PM_CUDA(e->upd_lat.ensure(n)); PM_CUDA(e->upd_lon.ensure(n));
    PM_CUDA(cudaMemcpyAsync(e->upd_lat.p, lat, (size_t)n * 8, cudaMemcpyHostToDevice, e->stream));
    PM_CUDA(cudaMemcpyAsync(e->upd_lon.p, lon, (size_t)n * 8, cudaMemcpyHostToDevice, e->stream));
  }
  pm::pm_scatter_rows<<<blocks_for(n, 256), 256, 0, e->stream>>>(e->wa.p, e->wb.p, lat ? e->lat.p : nullptr, lat ? e->lon.p : nullptr,
                                                                 e->scratch_idx.p, e->upd_a.p, e->upd_b.p, e->upd_lat.p, e->upd_lon.p, n,
                                                                 e->n_workers);
  PM_LAUNCH_CHECK("pm_scatter_rows");
  e->workers_checked = false;
  e->nacc_valid = false;
  e->matched = e->local_done = false;
  return PM_OK;
} catch (...) { return pm_guard_rc(); }

uint64_t pm_table_version(const pm_engine* e) { return e ? e->table_version : 0; }

// A second engine on the same device with the same configuration and its own stream and tables.
int pm_create_sibling(const pm_engine* e, pm_engine** out) try {
  if (!e || !out) return PM_E_INVALID;
  pm_cfg c = e->cfg;
  c.stream = nullptr;
  c.shard_first = c.shard_count = 0;
  return pm_create(&c, out);
} catch (...) { return pm_guard_rc(); }

// ------------------------------------------------------------------ evaluation
// Fast predicate only when both tables fit its operand limits; decided per match.
static int decide_fast(pm_engine* e, bool* fast) {
  *fast = false;
  if (e->tune_generic || !e->asks_small) return PM_OK;
  if (!e->workers_checked) {
    static const uint32_t ones[2] = {1u, 1u};
    PM_CUDA(cudaMemcpyAsync(e->counters.p + 2, ones, 8, cudaMemcpyHostToDevice, e->stream));
    if (e->n_workers) {
      pm::pm_check_worker_ranges<<<blocks_for(e->n_workers, 256), 256, 0, e->stream>>>(e->wa.p, e->wb.p, e->n_workers, e->counters.p + 2,
                                                                                       e->counters.p + 3);
      PM_LAUNCH_CHECK("pm_check_worker_ranges");
    }
    PM_CUDA(cudaMemcpyAsync(e->h_scalars.p + 4, e->counters.p + 2, 8, cudaMemcpyDeviceToHost, e->stream));
    PM_CUDA(cudaStreamSynchronize(e->stream));
    e->workers_small = e->h_scalars.p[4] != 0;
    e->prices_narrow = e->h_scalars.p[5] != 0;
    e->workers_checked = true;
  }
  *fast = e->workers_small;
  return PM_OK;
}

// FastRow.wp follows the model table: (re)bound after either table changed
static int bind_rows(pm_engine* e, bool wm) {
  if (e->rows_bound && e->rows_bound_wm == wm) return PM_OK;
  if (e->n_asks) {
    pm::pm_bind_rows<<<blocks_for(e->n_asks, 256), 256, 0, e->stream>>>(e->frows.p, e->opts_fast.p, wm ? e->bits_wm.p : e->bits.p,
                                                                        wm ? 1u : e->words, e->n_asks);
    PM_LAUNCH_CHECK("pm_bind_rows");
  }
  e->rows_bound = true;
  e->rows_bound_wm = wm;
  return PM_OK;
}

// More distinct model strings than the shared-memory acceptance table holds (BITS == 0: one global-memory lookup per
// (row, worker) pair, build kernel at 0.64 of the copy peak with 100k strings): turn the table around.  With at most 30
// patterns a worker's acceptance over ALL of them is one word, computed once per table change; the kernels then run
// their one-word form (BITS == 2) with the roles of row and worker swapped (EvalParams::nacc).  Fast predicate only.
static int worker_major(pm_engine* e, pm::EvalParams* p, int* bits_mode) {
  if (!e->nacc_valid) {
    PM_CUDA(e->nacc.ensure(std::max<uint32_t>(e->n_workers, 1)));
    PM_CUDA(e->bits_wm.ensure(32));
    uint32_t host[32];
    for (uint32_t r = 0; r < 32; ++r) host[r] = ~(1u << r);
    PM_CUDA(cudaMemcpyAsync(e->bits_wm.p, host, sizeof host, cudaMemcpyHostToDevice, e->stream));
    PM_CUDA(cudaStreamSynchronize(e->stream));   // `host` is a local
    if (e->n_workers) {
      pm::pm_worker_nacc<<<blocks_for(e->n_workers, 256), 256, 0, e->stream>>>(e->wa.p, e->bits.p, e->words, p->n_bits_rows, e->n_workers, e->nacc.p);
      PM_LAUNCH_CHECK("pm_worker_nacc");
    }
    e->nacc_valid = true;
  }
  p->bits = e->bits_wm.p;
  p->words = 1;
  p->nacc = e->nacc.p;
  *bits_mode = 2;
  return PM_OK;
}

// Does launch_build run the FastRow kernel (pm_build_cost_fast) for this table shape?  Only that kernel has the 16-bit
// form; PM_TUNE_BUILD=1 (staged-CSR kernel) and, with one-word acceptance rows, 3 / 4 (its occupancy variants) keep int64.
static bool fastrow_build(const pm_engine* e, bool fast, int bits_mode) {
  return fast && e->tune_build != 1 && !(bits_mode == 2 && (e->tune_build == 3 || e->tune_build == 4));
}

// The cost tile holds 16-bit price words (2 B per evaluation instead of 8) when the FastRow kernel runs and every worker
// price fits below the infeasible word 0xFFFF (decide_fast checked it); PM_TUNE_COST=8 forces the int64 tile.
static bool narrow_cost(const pm_engine* e, bool fast, int bits_mode) {
  return fastrow_build(e, fast, bits_mode) && e->prices_narrow && e->tune_cost != 8;
}

// `tile`: nt rows of ld words, int64 keys or (narrow) 16-bit price words
static void launch_build(pm_engine* e, const pm::EvalParams& p, int bits_mode, bool fast, bool narrow, dim3 grid,
                         uint32_t t0, uint32_t nt, uint32_t w0, uint32_t nw, size_t ld, void* tile) {
  long long* const cost = static_cast<long long*>(tile);
  uint16_t* const cost16 = static_cast<uint16_t*>(tile);
#define PM_BUILD_CASE(B, F) pm::pm_build_cost<B, F><<<grid, pm::kEvalThreads, 0, e->stream>>>(p, t0, nt, w0, nw, cost, ld)
#define PM_FAST_CASE(B, R)                                                                                           \
  if (narrow) pm::pm_build_cost_fast<B, R, uint16_t><<<grid, pm::kEvalThreads, 0, e->stream>>>(p, t0, nt, w0, nw, cost16, ld); \
  else pm::pm_build_cost_fast<B, R><<<grid, pm::kEvalThreads, 0, e->stream>>>(p, t0, nt, w0, nw, cost, ld)
  if (fast && bits_mode == 2 && e->tune_build == 3) {
    pm::pm_build_cost<2, true, 3><<<grid, pm::kEvalThreads, 0, e->stream>>>(p, t0, nt, w0, nw, cost, ld);
  } else if (fast && bits_mode == 2 && e->tune_build == 4) {
    pm::pm_build_cost<2, true, 4><<<grid, pm::kEvalThreads, 0, e->stream>>>(p, t0, nt, w0, nw, cost, ld);
  } else if (fast && e->tune_build != 1) {   // the round-2 kernel; PM_TUNE_BUILD=1 keeps the staged-CSR form for A/B runs
    // one-word acceptance rows are bound into the FastRows (pm_bind_rows) however many rows there are
    if (p.words == 1) bits_mode = 2;
    if (bits_mode == 2 && e->tune_build == 5) {          // rows-per-CTA experiments (profiles/)
      grid.y = blocks_for(nt, 128);
      PM_FAST_CASE(2, 128);
    } else if (bits_mode == 2 && e->tune_build == 6) {
      grid.y = blocks_for(nt, 256);
      PM_FAST_CASE(2, 256);
    } else {
      grid.y = blocks_for(nt, pm::kFastRows);
      if (bits_mode == 2) { PM_FAST_CASE(2, pm::kFastRows); }
      else if (bits_mode == 1) { PM_FAST_CASE(1, pm::kFastRows); }
      else { PM_FAST_CASE(0, pm::kFastRows); }
    }
  } else if (fast) {
    if (bits_mode == 2) PM_BUILD_CASE(2, true); else if (bits_mode == 1) PM_BUILD_CASE(1, true); else PM_BUILD_CASE(0, true);
  } else {
    if (bits_mode == 2) PM_BUILD_CASE(2, false); else if (bits_mode == 1) PM_BUILD_CASE(1, false); else PM_BUILD_CASE(0, false);
  }
#undef PM_FAST_CASE
#undef PM_BUILD_CASE
}

static void launch_fused(pm_engine* e, const pm::EvalParams& p, int bits_mode, bool fast, bool stats, dim3 grid,
                         uint32_t t0, uint32_t nt, uint32_t w0, uint32_t nw) {
#define PM_FUSED_CASE(B, F, S) pm::pm_fused_eval<B, F, S><<<grid, pm::kEvalThreads, 0, e->stream>>>(p, t0, nt, w0, nw, e->first_ask.p, e->ask_best.p, e->ask_count.p)
  if (fast && !stats && bits_mode == 2) { PM_FUSED_CASE(2, true, false); return; }   // the lean common case
  if (fast) {
    if (bits_mode == 2) PM_FUSED_CASE(2, true, true); else if (bits_mode == 1) PM_FUSED_CASE(1, true, true); else PM_FUSED_CASE(0, true, true);
  } else {
    if (bits_mode == 2) PM_FUSED_CASE(2, false, true); else if (bits_mode == 1) PM_FUSED_CASE(1, false, true); else PM_FUSED_CASE(0, false, true);
  }
#undef PM_FUSED_CASE
}

static void launch_argmin(pm_engine* e, bool narrow, size_t ld, uint32_t nt, uint32_t t0, uint32_t w0, uint32_t nw) {
#define PM_ARGMIN16_CASE(S, RPW)                                                                                      \
  {                                                                                                                   \
    dim3 grid(blocks_for(ld, (S) * 256 * pm::kArgWarps), blocks_for(nt, pm::kArgRows));                               \
    pm::pm_argmin16<S, RPW><<<grid, pm::kArgThreads, 0, e->stream>>>(reinterpret_cast<const uint16_t*>(e->cost.p), ld, \
                                                                     nt, t0, w0, nw, e->first_ask.p, e->ask_best.p,  \
                                                                     e->ask_count.p);                                 \
  }
  if (narrow) {   // PM_TUNE_ARGMIN picks the shape of the 16-bit kernel here (profiles/r03_argmin16_shapes.txt)
    switch (e->tune_argmin) {
      case 1: PM_ARGMIN16_CASE(2, 4) break;
      case 2: PM_ARGMIN16_CASE(4, 1) break;
      case 3: PM_ARGMIN16_CASE(8, 1) break;
      case 4: PM_ARGMIN16_CASE(4, 4) break;
      case 5: PM_ARGMIN16_CASE(8, 2) break;
      default: PM_ARGMIN16_CASE(4, 2) break;
    }
    return;
  }
#undef PM_ARGMIN16_CASE
#define PM_ARGMIN_CASE(S, RPW)                                                                      \
  {                                                                                                  \
    dim3 grid(blocks_for(ld, (S) * 64 * pm::kArgWarps), blocks_for(nt, pm::kArgRows));                               \
    pm::pm_argmin<S, RPW><<<grid, pm::kArgThreads, 0, e->stream>>>(reinterpret_cast<const long long*>(e->cost.p), ld, \
                                                                   nt, t0, w0, nw, e->first_ask.p, e->ask_best.p,    \
                                                                   e->ask_count.p);                 \
  }
  switch (e->tune_argmin) {
    case 1: PM_ARGMIN_CASE(4, 1) break;
    case 2: PM_ARGMIN_CASE(4, 2) break;
    case 3: PM_ARGMIN_CASE(8, 2) break;
    case 4: PM_ARGMIN_CASE(4, 4) break;
    case 5: PM_ARGMIN_CASE(8, 1) break;
    case 6: PM_ARGMIN_CASE(8, 4) break;
    case 7: PM_ARGMIN_CASE(16, 1) break;
    case 8: PM_ARGMIN_CASE(16, 2) break;
    default: PM_ARGMIN_CASE(8, 2) break;
  }
#undef PM_ARGMIN_CASE
}

static int match_local_locked(pm_engine* e, uint32_t mode) {
  if (!e->have_workers || !e->have_asks) return e->fail(PM_E_STATE, "pm_match: worker and ask tables must be set first");
  if (e->max_pattern_row > e->n_patterns || (e->max_pattern_row && !e->have_bits))
    return e->fail(PM_E_STATE, "pm_match: an ask references a model pattern missing from the model table");
  const uint32_t base_mode = mode & 0xFFu;
  if (base_mode == PM_MODE_AUCTION) return e->fail(PM_E_INVALID, "pm_match: auction mode goes through pm_match");
  if (base_mode != PM_MODE_FIRST_FIT && base_mode != PM_MODE_PROXIMITY && base_mode != PM_MODE_PROXIMITY_MERGE)
    return e->fail(PM_E_INVALID, "pm_match: unknown mode");
  if ((base_mode == PM_MODE_PROXIMITY && !e->all_solo) || base_mode == PM_MODE_PROXIMITY_MERGE) {
    if (!e->have_loc) return e->fail(PM_E_STATE, "pm_match: proximity mode needs pm_set_worker_locations");
    if (e->any_max_zero)
      return e->fail(PM_E_UNSUPPORTED, "pm_match: max_group_size == 0 is not supported in proximity mode");
  }
  PM_CUDA(cudaSetDevice(e->device));
  const uint32_t W = e->n_workers, T = e->n_asks;
  uint32_t w0 = 0, nw = 0;
  e->shard(&w0, &nw);
  if ((uint64_t)w0 + nw > W) return e->fail(PM_E_INVALID, "pm_match: shard range exceeds the worker table");
  if (!e->have_bits) {  // tables without any model clause: a one-row all-ones table
    PM_CUDA(e->bits.ensure(1));
    PM_CUDA(cudaMemsetAsync(e->bits.p, 0xFF, 4, e->stream));
    e->words = 1;
  }

  e->stats = pm_stats{};
  e->ev_pending.clear();
  e->ev_used = 0;
  const bool timing = (e->cfg.flags & PM_CFG_TIMING) != 0;
  if (timing) PM_CUDA(cudaEventRecord(e->ev0, e->stream));

  PM_CUDA(e->first_ask.ensure(W));
  PM_CUDA(e->ask_best.ensure(T));
  PM_CUDA(e->ask_count.ensure(T));
  PM_CUDA(cudaMemsetAsync(e->first_ask.p, 0xFF, (size_t)std::max<uint32_t>(W, 1) * 4, e->stream));
  PM_CUDA(cudaMemsetAsync(e->ask_count.p, 0, (size_t)std::max<uint32_t>(T, 1) * 4, e->stream));
  if (T) {
    pm::pm_fill_i64<<<std::min(blocks_for(T, 256), 1184u), 256, 0, e->stream>>>(e->ask_best.p, pm::kInf, T);
    PM_LAUNCH_CHECK("pm_fill_i64");
  }

  if (T && nw) {
    pm::EvalParams p = eval_params(e);
    int bits_mode = ((uint64_t)p.n_bits_rows * p.words <= (uint64_t)pm::kBitsCap) ? (p.words == 1 ? 2 : 1) : 0;
    bool fast = false;
    {
      int rc = decide_fast(e, &fast);
      if (rc != PM_OK) return rc;
    }
    const bool wm = fast && bits_mode == 0 && p.n_bits_rows <= 31u && e->tune_build != 7;   // PM_TUNE_BUILD=7: keep the global-memory table
    if (wm) {
      const int rc = worker_major(e, &p, &bits_mode);
      if (rc != PM_OK) return rc;
    }
    if (mode & PM_PATH_FUSED) {
      Timer tm(e, &e->stats.ms_fused);
      const uint32_t rows_per_launch = 65535u * pm::kEvalRows;
      for (uint32_t t0 = 0; t0 < T; t0 += rows_per_launch) {
        const uint32_t nt = std::min(rows_per_launch, T - t0);
        dim3 grid(blocks_for(nw, pm::kEvalCols), blocks_for(nt, pm::kEvalRows));
        launch_fused(e, p, bits_mode, fast, (mode & PM_NO_ASK_STATS) == 0, grid, t0, nt, w0, nw);
        PM_LAUNCH_CHECK("pm_fused_eval");
        ++e->stats.n_fused_launches;
      }
      tm.stop();
      e->stats.n_tiles = 1;
    } else {
      // leading dimension = whole CTA stripes of the build kernel (1024 columns): its stores need no bounds test;
      // the columns past the shard hold "infeasible" and cost 0.05 % of a 1M-worker row
      const size_t ld = (((size_t)nw + pm::kEvalCols - 1) / pm::kEvalCols) * pm::kEvalCols;
      {
        const int rc = bind_rows(e, wm);
        if (rc != PM_OK) return rc;
      }
      const bool narrow = narrow_cost(e, fast, bits_mode);
      const size_t word_bytes = narrow ? 2 : 8;    // 16-bit price words or int64 keys
      // rows per tile as the int64 tile has them, whatever the width: both widths run the same tile sequence (the A/B
      // differs in the word alone) and the 16-bit tile takes a quarter of the budget.  Taller 16-bit tiles were faster on
      // cfg3 (4096 rows: 7 %, profiles/r03_cost_width_ab_4096_rows.txt)
      uint64_t rows = e->cfg.cost_tile_bytes / (ld * 8);
      if (rows == 0) rows = 1;
      rows = std::min<uint64_t>(rows, T);
      rows = std::min<uint64_t>(rows, 65535ull * pm::kArgRows);
      if (rows >= 1024) rows &= ~(uint64_t)511;   // whole row bands of the build kernel (no ragged last band in every tile)
      cudaError_t ce = e->cost.ensure((size_t)rows * ld * word_bytes);
      if (ce != cudaSuccess) {
        cudaGetLastError();
        return e->fail(PM_E_NOMEM, "pm_match: cannot allocate the cost tile; lower pm_cfg.cost_tile_bytes");
      }
      for (uint32_t t0 = 0; t0 < T; t0 += (uint32_t)rows) {
        const uint32_t nt = (uint32_t)std::min<uint64_t>(rows, T - t0);
        {
          Timer tm(e, &e->stats.ms_build);
          dim3 grid(blocks_for(ld, pm::kEvalCols), blocks_for(nt, pm::kEvalRows));
          launch_build(e, p, bits_mode, fast, narrow, grid, t0, nt, w0, nw, ld, e->cost.p);
          PM_LAUNCH_CHECK("pm_build_cost");
          tm.stop();
          ++e->stats.n_build_launches;
        }
        {
          Timer tm(e, &e->stats.ms_argmin);
          launch_argmin(e, narrow, ld, nt, t0, w0, nw);
          PM_LAUNCH_CHECK("pm_argmin");
          tm.stop();
          ++e->stats.n_argmin_launches;
        }
        ++e->stats.n_tiles;
        // algorithmic: 2 or 8 B per evaluation (padding columns not counted)
        e->stats.cost_bytes_written += (uint64_t)nt * nw * word_bytes;
        e->stats.cost_bytes_read += (uint64_t)nt * nw * word_bytes;
      }
    }
    e->stats.evals = (uint64_t)T * nw;
  }
  e->local_done = true;
  e->matched = false;
  return PM_OK;
}

// ------------------------------------------------------------------ resolution
static int sort_and_scan(pm_engine* e, uint32_t n_bins, uint32_t shift) {
  const uint32_t W = e->n_workers;
  PM_CUDA(cudaMemsetAsync(e->hist.p, 0, ((size_t)n_bins + 1) * 4, e->stream));
  if (W) {
    pm::pm_make_keys<<<blocks_for(W, 256), 256, 0, e->stream>>>(e->first_ask.p, e->wa.p, W, shift, e->keys.p, e->hist.p);
    PM_LAUNCH_CHECK("pm_make_keys");
  }
  size_t tmp_scan = 0, tmp_sort = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, tmp_scan, e->hist.p, e->seg_start.p, (int)(n_bins + 1), e->stream);
  cub::DeviceRadixSort::SortPairs(nullptr, tmp_sort, e->keys.p, e->keys_sorted.p, e->iota.p, e->order.p, (int)W, 0, 32, e->stream);
  size_t tmp = std::max(tmp_scan, tmp_sort);
  PM_CUDA(e->cub_tmp.ensure(tmp));
  PM_CUDA(cub::DeviceScan::ExclusiveSum(e->cub_tmp.p, tmp, e->hist.p, e->seg_start.p, (int)(n_bins + 1), e->stream));
  if (W) PM_CUDA(cub::DeviceRadixSort::SortPairs(e->cub_tmp.p, tmp, e->keys.p, e->keys_sorted.p, e->iota.p, e->order.p, (int)W, 0, 32, e->stream));
  return PM_OK;
}

// The O(W + T) resolution sweep.  Everything between the sort and the last kernel stays on the device (counts are
// read through device pointers, tables are sized for the worst case), so a pass has exactly ONE host synchronisation:
// the one at the end that brings back {groups, members, bumped} (and resolves the event timers).
static int match_finish_locked(pm_engine* e, uint32_t mode) {
  if (!e->local_done) return e->fail(PM_E_STATE, "pm_match_finish: pm_match_local has not run");
  PM_CUDA(cudaSetDevice(e->device));
  const uint32_t base_mode = mode & 0xFFu;
  const uint32_t W = e->n_workers, T = e->n_asks;
  const bool merge_mode = base_mode == PM_MODE_PROXIMITY_MERGE;
  const bool prox_general = (base_mode == PM_MODE_PROXIMITY && !e->all_solo) || merge_mode;
  const uint32_t shift = (base_mode == PM_MODE_PROXIMITY && !prox_general) ? 1u : 0u;
  const uint32_t n_bins = T << shift;
  Timer tm(e, &e->stats.ms_resolve);

  PM_CUDA(e->keys.ensure(W)); PM_CUDA(e->keys_sorted.ensure(W)); PM_CUDA(e->iota.ensure(W));
  PM_CUDA(e->order.ensure(W)); PM_CUDA(e->hist.ensure((size_t)n_bins + 1));
  PM_CUDA(e->seg_start.ensure((size_t)n_bins + 1)); PM_CUDA(e->ngroups.ensure((size_t)n_bins + 1));
  PM_CUDA(e->group_base.ensure((size_t)n_bins + 1));
  PM_CUDA(e->worker_group.ensure(W)); PM_CUDA(e->worker_ask.ensure(W)); PM_CUDA(e->members.ensure(W));
  PM_CUDA(cudaMemsetAsync(e->counters.p, 0, 12 * 4, e->stream));   // [12..13] belong to pm_set_asks
  if (W) {
    pm::pm_iota_u32<<<std::min(blocks_for(W, 256), 1184u), 256, 0, e->stream>>>(e->iota.p, W);
    PM_LAUNCH_CHECK("pm_iota_u32");
  }
  int rc = sort_and_scan(e, n_bins, shift);
  if (rc != PM_OK) return rc;
  uint32_t* const scal = e->counters.p + 8;   // device mailbox {groups, members, bumped, overflow}
  bool prox_grid_ran = false;

  if (prox_general) {
    // sequential-per-group nearest-neighbour formation (pm_proximity.cuh)
    uint32_t P = 1;
    while (P < std::max<uint32_t>(W, 1)) P <<= 1;
    const uint32_t cap = W + T + 1;
    PM_CUDA(e->base_len.ensure(T)); PM_CUDA(e->xhead.ensure(T)); PM_CUDA(e->xcount.ensure(T));
    PM_CUDA(e->xnext.ensure(W)); PM_CUDA(e->popped.ensure(W));
    PM_CUDA(e->prox_list.ensure(W)); PM_CUDA(e->prox_xs.ensure(P)); PM_CUDA(e->prox_dist.ensure(W));
    PM_CUDA(e->members_raw.ensure(W));
    PM_CUDA(e->group_ask.ensure((size_t)cap + 1)); PM_CUDA(e->group_off.ensure((size_t)cap + 1));
    PM_CUDA(cudaMemcpyAsync(e->base_len.p, e->hist.p, (size_t)T * 4, cudaMemcpyDeviceToDevice, e->stream));
    PM_CUDA(cudaMemsetAsync(e->xhead.p, 0xFF, (size_t)T * 4, e->stream));
    PM_CUDA(cudaMemsetAsync(e->xcount.p, 0, (size_t)T * 4, e->stream));
    PM_CUDA(cudaMemsetAsync(e->worker_group.p, 0xFF, (size_t)std::max<uint32_t>(W, 1) * 4, e->stream));
    PM_CUDA(cudaMemsetAsync(e->worker_ask.p, 0xFF, (size_t)std::max<uint32_t>(W, 1) * 4, e->stream));
    pm::ProxParams pp;
    pp.ev = eval_params(e);
    pp.lat = e->lat.p; pp.lon = e->lon.p;
    pp.cur = e->first_ask.p; pp.base_len = e->base_len.p; pp.seg_start = e->seg_start.p; pp.order = e->order.p;
    pp.xhead = e->xhead.p; pp.xnext = e->xnext.p; pp.xcount = e->xcount.p; pp.amin = e->amin.p; pp.amax = e->amax.p;
    pp.list = e->prox_list.p; pp.xs = e->prox_xs.p; pp.dist = e->prox_dist.p; pp.popped = e->popped.p;
    pp.worker_group = e->worker_group.p; pp.worker_ask = e->worker_ask.p; pp.group_ask = e->group_ask.p;
    pp.group_off = e->group_off.p; pp.members = e->members_raw.p; pp.out_counts = scal;   // {G, M, bumped, overflow}
    pp.group_cap = cap;
    if (e->coop_blocks < 0) {   // once per engine: can the whole-chip sweep be launched cooperatively, and how wide?
      int coop = 0, per_sm = 0, sms = 0;
      cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, e->device);
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->device);
      if (coop && cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pm::pm_proximity_grid, pm::kPgThreads, 0) == cudaSuccess)
        e->coop_blocks = per_sm * sms;
      else
        e->coop_blocks = 0;
      (void)cudaGetLastError();
    }
    if (merge_mode) pm::pm_merge_sweep<<<1, pm::kProxThreads, 0, e->stream>>>(pp);
    else if (e->tune_prox == 0 && e->coop_blocks > 0) {
      // all SMs: one grid barrier per group instead of one CTA doing everything (pm_proximity_grid.cuh)
      const unsigned grid = std::max(1u, std::min<unsigned>((unsigned)e->coop_blocks, blocks_for(std::max<uint32_t>(W, 1), pm::kPgThreads)));
      PM_CUDA(e->pg_part_d.ensure((size_t)2 * grid * pm::kPgTopK)); PM_CUDA(e->pg_part_i.ensure((size_t)2 * grid * pm::kPgTopK));
      PM_CUDA(e->pg_cta_cnt.ensure((size_t)2 * grid)); PM_CUDA(e->pg_ctl.ensure(8));
      PM_CUDA(e->pg_clat.ensure(W)); PM_CUDA(e->pg_clon.ensure(W)); PM_CUDA(e->pg_ccos.ensure(W));
      PM_CUDA(cudaMemsetAsync(e->pg_ctl.p, 0, 32, e->stream));
      pm::GridProxParams gp;
      gp.p = pp;
      gp.part_d = e->pg_part_d.p; gp.part_i = e->pg_part_i.p; gp.cta_cnt = e->pg_cta_cnt.p; gp.gctl = e->pg_ctl.p;
      gp.clat = e->pg_clat.p; gp.clon = e->pg_clon.p; gp.ccos = e->pg_ccos.p;
      gp.n_workers = W;
      void* args[] = {&gp};
      PM_CUDA(cudaLaunchCooperativeKernel((const void*)pm::pm_proximity_grid, dim3(grid), dim3(pm::kPgThreads), args, 0, e->stream));
      PM_CUDA(cudaMemcpyAsync(e->h_scalars.p + 24, e->pg_ctl.p + 4, 12, cudaMemcpyDeviceToHost, e->stream));
      prox_grid_ran = true;
    }
    else if (e->tune_prox & 1) {   // experimental: same groups from a latitude-ordered view (pm_proximity_band.cuh)
      PM_CUDA(e->prox_lat_key.ensure(P)); PM_CUDA(e->prox_lat_ord.ensure(P)); PM_CUDA(e->prox_rank_of.ensure(W));
      pm::BandParams bp;
      bp.p = pp;
      bp.lat_key = e->prox_lat_key.p; bp.lat_ord = e->prox_lat_ord.p; bp.rank_of = e->prox_rank_of.p;
      pm::pm_proximity_sweep_banded<<<1, pm::kProxThreads, 0, e->stream>>>(bp);
    }
    else pm::pm_proximity_sweep<<<1, pm::kProxThreads, 0, e->stream>>>(pp);
    PM_LAUNCH_CHECK("pm_proximity_sweep");
    if (W) {
      pm::pm_order_members<<<blocks_for(W, 256), 256, 0, e->stream>>>(
          e->members_raw.p, scal + 1, e->worker_group.p, e->group_off.p, e->have_rank ? e->addr_rank.p : nullptr, e->members.p);
      PM_LAUNCH_CHECK("pm_order_members");
    }
  } else {
    if (shift == 0 && T && !e->all_solo) {
      // under-filled tails: flagged on the device; the single-CTA sweep returns at once when there is none
      pm::pm_check_tails<<<blocks_for(T, 256), 256, 0, e->stream>>>(e->hist.p, e->amin.p, e->amax.p, T, e->counters.p);
      PM_LAUNCH_CHECK("pm_check_tails");
      PM_CUDA(e->base_len.ensure(T)); PM_CUDA(e->xhead.ensure(T)); PM_CUDA(e->xcount.ensure(T));
      PM_CUDA(e->xnext.ensure(W)); PM_CUDA(e->popped.ensure(W));
      PM_CUDA(cudaMemcpyAsync(e->base_len.p, e->hist.p, (size_t)T * 4, cudaMemcpyDeviceToDevice, e->stream));
      PM_CUDA(cudaMemsetAsync(e->xhead.p, 0xFF, (size_t)T * 4, e->stream));
      PM_CUDA(cudaMemsetAsync(e->xcount.p, 0, (size_t)T * 4, e->stream));
      pm::SweepParams sp;
      sp.ev = eval_params(e);
      sp.cur = e->first_ask.p; sp.base_len = e->base_len.p; sp.seg_start = e->seg_start.p;
      sp.order = e->order.p; sp.xhead = e->xhead.p; sp.xnext = e->xnext.p; sp.xcount = e->xcount.p;
      sp.amin = e->amin.p; sp.amax = e->amax.p; sp.popped = e->popped.p; sp.n_bumped = e->counters.p + 1;
      sp.any_bad = e->counters.p;
      pm::pm_sweep<<<1, 1024, 0, e->stream>>>(sp);
      PM_LAUNCH_CHECK("pm_sweep");
      rc = sort_and_scan(e, n_bins, shift);   // owners may have moved
      if (rc != PM_OK) return rc;
    }

    if (n_bins) {
      pm::pm_count_groups<<<blocks_for(n_bins, 256), 256, 0, e->stream>>>(e->hist.p, e->amin.p, e->amax.p, n_bins, shift, e->ngroups.p);
      PM_LAUNCH_CHECK("pm_count_groups");
    }
    PM_CUDA(cudaMemsetAsync(e->ngroups.p + n_bins, 0, 4, e->stream));
    {
      size_t tmp = 0;
      cub::DeviceScan::ExclusiveSum(nullptr, tmp, e->ngroups.p, e->group_base.p, (int)(n_bins + 1), e->stream);
      PM_CUDA(e->cub_tmp.ensure(tmp));
      PM_CUDA(cub::DeviceScan::ExclusiveSum(e->cub_tmp.p, tmp, e->ngroups.p, e->group_base.p, (int)(n_bins + 1), e->stream));
    }
    // groups <= members + one empty group per bin; sized for that so the count never has to visit the host first
    const size_t gcap = (size_t)W + n_bins + 1;
    PM_CUDA(e->group_ask.ensure(gcap + 1));
    PM_CUDA(e->group_off.ensure(gcap + 1));
    const uint32_t* n_assigned_dev = e->seg_start.p + n_bins;
    PM_CUDA(cudaMemsetAsync(e->worker_group.p, 0xFF, (size_t)std::max<uint32_t>(W, 1) * 4, e->stream));
    PM_CUDA(cudaMemsetAsync(e->worker_ask.p, 0xFF, (size_t)std::max<uint32_t>(W, 1) * 4, e->stream));
    if (W) {
      pm::pm_emit_workers<<<blocks_for(W, 256), 256, 0, e->stream>>>(
          e->keys_sorted.p, e->order.p, n_assigned_dev, e->hist.p, e->seg_start.p, e->group_base.p, e->amin.p,
          e->amax.p, shift, e->worker_group.p, e->worker_ask.p, e->group_ask.p, e->group_off.p);
      PM_LAUNCH_CHECK("pm_emit_workers");
    }
    if (n_bins && !e->all_solo) {
      pm::pm_emit_empty_groups<<<blocks_for(n_bins, 256), 256, 0, e->stream>>>(
          e->hist.p, e->seg_start.p, e->group_base.p, e->ngroups.p, e->amin.p, n_bins, shift, e->group_ask.p, e->group_off.p);
      PM_LAUNCH_CHECK("pm_emit_empty_groups");
    }
    pm::pm_close_groups<<<1, 1, 0, e->stream>>>(e->group_base.p + n_bins, n_assigned_dev, e->counters.p + 1, e->group_off.p, scal);
    PM_LAUNCH_CHECK("pm_close_groups");
    if (W) {
      pm::pm_order_members<<<blocks_for(W, 256), 256, 0, e->stream>>>(
          e->order.p, n_assigned_dev, e->worker_group.p, e->group_off.p, e->have_rank ? e->addr_rank.p : nullptr, e->members.p);
      PM_LAUNCH_CHECK("pm_order_members");
    }
  }
  tm.stop();
  PM_CUDA(cudaMemcpyAsync(e->h_scalars.p + 8, scal, 16, cudaMemcpyDeviceToHost, e->stream));
  if (e->cfg.flags & PM_CFG_TIMING) PM_CUDA(cudaEventRecord(e->ev1, e->stream));
  PM_CUDA(cudaStreamSynchronize(e->stream));   // the pass's one host synchronisation
  if (prox_general && e->h_scalars.p[11]) return e->fail(PM_E_CUDA, "pm_match: proximity group table overflow");
  e->n_groups = e->h_scalars.p[8];
  e->n_assigned = e->h_scalars.p[9];
  e->stats.n_bumped = e->h_scalars.p[10];
  if (prox_grid_ran) {   // cooperative proximity sweep: seed-parallel batches, groups formed in them, groups formed one at a time
    e->stats.n_tiles = e->h_scalars.p[24];
    e->stats.n_rounds = e->h_scalars.p[25];
    e->stats.n_build_launches = e->h_scalars.p[26];
  }
  if (e->cfg.flags & PM_CFG_TIMING) {
    PM_CUDA(cudaEventElapsedTime(&e->stats.ms_total, e->ev0, e->ev1));
    e->resolve_timers();
  }
  e->matched = true;
  return PM_OK;
}

// ------------------------------------------------------------------ extension: auction
// Ask classes for the auction: asks with identical requirement rows (pm_auction.cuh).
static int auction_build_classes(pm_engine* e) {
  const uint32_t T = e->n_asks;
  e->auc_n_classes = 0;
  PM_CUDA(e->auc_class_of.ensure(T)); PM_CUDA(e->auc_class_rep.ensure(T)); PM_CUDA(e->auc_hash.ensure(T));
  PM_CUDA(e->auc_hash_out.ensure(T)); PM_CUDA(e->auc_idx.ensure(T)); PM_CUDA(e->auc_sorted.ensure(T));
  PM_CUDA(e->auc_flag.ensure((size_t)T + 1)); PM_CUDA(e->auc_incl.ensure(T));
  if (T == 0) { e->auc_classes_valid = true; return PM_OK; }
  pm::pm_auction_ask_hash<<<blocks_for(T, 256), 256, 0, e->stream>>>(e->asks.p, e->opts.p, e->have_min_rep ? e->ask_min_rep.p : nullptr, T, e->auc_hash.p, e->auc_idx.p);
  PM_LAUNCH_CHECK("pm_auction_ask_hash");
  size_t tmp_sort = 0, tmp_scan = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, tmp_sort, e->auc_hash.p, e->auc_hash_out.p, e->auc_idx.p, e->auc_sorted.p, (int)T, 0, 64, e->stream);
  cub::DeviceScan::InclusiveSum(nullptr, tmp_scan, e->auc_flag.p, e->auc_incl.p, (int)T, e->stream);
  size_t tmp = std::max(tmp_sort, tmp_scan);
  PM_CUDA(e->cub_tmp.ensure(tmp));
  PM_CUDA(cub::DeviceRadixSort::SortPairs(e->cub_tmp.p, tmp, e->auc_hash.p, e->auc_hash_out.p, e->auc_idx.p, e->auc_sorted.p, (int)T, 0, 64, e->stream));
  pm::pm_auction_class_flags<<<blocks_for(T, 256), 256, 0, e->stream>>>(e->asks.p, e->opts.p, e->have_min_rep ? e->ask_min_rep.p : nullptr, e->auc_sorted.p, T, e->auc_flag.p);
  PM_LAUNCH_CHECK("pm_auction_class_flags");
  PM_CUDA(cub::DeviceScan::InclusiveSum(e->cub_tmp.p, tmp, e->auc_flag.p, e->auc_incl.p, (int)T, e->stream));
  pm::pm_auction_class_assign<<<blocks_for(T, 256), 256, 0, e->stream>>>(e->auc_sorted.p, e->auc_flag.p, e->auc_incl.p, T,
                                                                          e->auc_class_of.p, e->auc_class_rep.p);
  PM_LAUNCH_CHECK("pm_auction_class_assign");
  PM_CUDA(cudaMemcpyAsync(e->h_scalars.p + 16, e->auc_incl.p + (T - 1), 4, cudaMemcpyDeviceToHost, e->stream));
  PM_CUDA(cudaStreamSynchronize(e->stream));
  e->auc_n_classes = e->h_scalars.p[16];
  e->auc_classes_valid = true;
  return PM_OK;
}

static int match_auction_locked(pm_engine* e) {
  if (!e->have_workers || !e->have_asks) return e->fail(PM_E_STATE, "pm_match: worker and ask tables must be set first");
  if (!e->have_caps) return e->fail(PM_E_STATE, "pm_match: auction mode needs pm_set_ask_price_caps");
  if (e->max_pattern_row > e->n_patterns || (e->max_pattern_row && !e->have_bits))
    return e->fail(PM_E_STATE, "pm_match: an ask references a model pattern missing from the model table");
  if (e->cfg.shard_count || e->comm) return e->fail(PM_E_UNSUPPORTED, "pm_match: auction mode is single-GPU");
  PM_CUDA(cudaSetDevice(e->device));
  const uint32_t W = e->n_workers, T = e->n_asks;
  if (!e->have_bits) {
    PM_CUDA(e->bits.ensure(1));
    PM_CUDA(cudaMemsetAsync(e->bits.p, 0xFF, 4, e->stream));
    e->words = 1;
  }
  e->stats = pm_stats{};
  e->ev_pending.clear();
  e->ev_used = 0;
  if (e->cfg.flags & PM_CFG_TIMING) PM_CUDA(cudaEventRecord(e->ev0, e->stream));
  Timer tm(e, &e->stats.ms_fused);
  if (!e->auc_classes_valid) {
    const int rc = auction_build_classes(e);
    if (rc != PM_OK) return rc;
  }
  const uint32_t C = e->auc_n_classes;
  constexpr unsigned kScanGrid = 296u;   // two scanning CTAs per SM (shared memory)
  PM_CUDA(e->auc_price.ensure((size_t)W + 2)); PM_CUDA(e->auc_owner.ensure(W)); PM_CUDA(e->auc_bid_max.ensure(W));
  PM_CUDA(e->auc_winner.ensure(W)); PM_CUDA(e->auc_assigned.ensure(T)); PM_CUDA(e->auc_withdrawn.ensure(T));
  PM_CUDA(e->auc_active.ensure((size_t)2 * std::max<uint32_t>(T, 1))); PM_CUDA(e->auc_bid_w.ensure(T)); PM_CUDA(e->auc_bid_p.ensure(T));
  PM_CUDA(e->auc_flag.ensure((size_t)T + 1)); PM_CUDA(e->auc_gidx.ensure((size_t)T + 1));
  PM_CUDA(e->auc_theta.ensure(C)); PM_CUDA(e->auc_theta_w.ensure(C)); PM_CUDA(e->auc_cand.ensure((size_t)C * pm::kAucCache));
  PM_CUDA(e->auc_pool.ensure((size_t)C * pm::kAucPool)); PM_CUDA(e->auc_pool_bound_v.ensure(C)); PM_CUDA(e->auc_pool_bound_w.ensure(C));
  PM_CUDA(e->auc_walk_list.ensure(C)); PM_CUDA(e->auc_split_v.ensure(kScanGrid * 16)); PM_CUDA(e->auc_split_w.ensure(kScanGrid * 16));
  PM_CUDA(e->auc_split_ticket.ensure(kScanGrid));
  PM_CUDA(cudaMemsetAsync(e->auc_split_ticket.p, 0, kScanGrid * 4, e->stream));
  PM_CUDA(e->auc_split_first.ensure(kScanGrid)); PM_CUDA(e->auc_skip_key.ensure(std::max<uint32_t>(C, 1)));
  PM_CUDA(cudaMemsetAsync(e->auc_split_first.p, 0xFF, kScanGrid * 4, e->stream));
  PM_CUDA(cudaMemsetAsync(e->auc_skip_key.p, 0, (size_t)std::max<uint32_t>(C, 1) * 8, e->stream));
  PM_CUDA(e->auc_class_req.ensure(C)); PM_CUDA(e->auc_class_list.ensure(C)); PM_CUDA(e->auc_retry.ensure(T)); PM_CUDA(e->auc_fallback.ensure(T));
  PM_CUDA(e->auc_perm.ensure((size_t)W + 4)); PM_CUDA(e->auc_pos_of.ensure(W));
  PM_CUDA(e->auc_idx.ensure(std::max(W, T))); PM_CUDA(e->auc_wa_s.ensure(W)); PM_CUDA(e->auc_wb_s.ensure(W)); PM_CUDA(e->auc_price_s.ensure((size_t)W + 2));
  PM_CUDA(e->auc_ctl.ensure(1)); PM_CUDA(e->h_ctl.ensure(1));
  PM_CUDA(e->worker_group.ensure(W)); PM_CUDA(e->worker_ask.ensure(W)); PM_CUDA(e->members.ensure(std::max(W, T)));
  PM_CUDA(e->group_ask.ensure((size_t)T + 1)); PM_CUDA(e->group_off.ensure((size_t)T + 2));
  PM_CUDA(e->ask_best.ensure(T)); PM_CUDA(e->ask_count.ensure(T)); PM_CUDA(e->first_ask.ensure(W));
  PM_CUDA(cudaMemsetAsync(e->auc_price.p, 0, ((size_t)W + 2) * 8, e->stream));
  PM_CUDA(cudaMemsetAsync(e->auc_price_s.p, 0, ((size_t)W + 2) * 8, e->stream));
  PM_CUDA(cudaMemsetAsync(e->auc_ctl.p, 0, sizeof(pm::AuctionCtl), e->stream));
  PM_CUDA(cudaMemsetAsync(e->auc_class_req.p, 0, (size_t)std::max<uint32_t>(C, 1) * 4, e->stream));
  PM_CUDA(e->auc_ckey.ensure(W)); PM_CUDA(e->auc_ckey_s.ensure(W));
  // `reputation` clause: only when a floor was given; a missing worker column is a column of zeros
  const bool use_rep = e->have_min_rep;
  if (use_rep) {
    if (!e->have_rep) {
      PM_CUDA(e->reputation.ensure(std::max<size_t>(e->wa.n, 1)));
      PM_CUDA(cudaMemsetAsync(e->reputation.p, 0, std::max<size_t>(e->wa.n, 1) * 4, e->stream));
      e->have_rep = true;
    }
    PM_CUDA(e->auc_rep_s.ensure((size_t)W + 4));
    PM_CUDA(cudaMemsetAsync(e->auc_rep_s.p, 0, ((size_t)W + 4) * 4, e->stream));
  }
  if (W) {
    pm::pm_fill_i64<<<std::min(blocks_for(W, 256), 1184u), 256, 0, e->stream>>>(e->auc_bid_max.p, pm::kAucNeg, W);
    PM_LAUNCH_CHECK("pm_fill_i64");
  }
  // worker planes sorted by (ask_price * S + price, index): stable radix sort; redone as prices move (below)
  auto sort_workers = [&]() -> int {
    if (!W) return PM_OK;
    pm::pm_auction_cost_keys<<<blocks_for(W, 256), 256, 0, e->stream>>>(e->wb.p, e->auc_price.p, (long long)e->auc_scale, W, reinterpret_cast<unsigned long long*>(e->auc_ckey.p), e->auc_idx.p);
    PM_LAUNCH_CHECK("pm_auction_cost_keys");
    size_t tmp = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tmp, e->auc_ckey.p, e->auc_ckey_s.p, e->auc_idx.p, e->auc_perm.p, (int)W, 0, 64, e->stream);
    PM_CUDA(e->cub_tmp.ensure(tmp));
    PM_CUDA(cub::DeviceRadixSort::SortPairs(e->cub_tmp.p, tmp, e->auc_ckey.p, e->auc_ckey_s.p, e->auc_idx.p, e->auc_perm.p, (int)W, 0, 64, e->stream));
    pm::pm_auction_gather_sorted<<<blocks_for(W, 256), 256, 0, e->stream>>>(e->wa.p, e->wb.p, e->auc_perm.p, e->auc_price.p, W, e->auc_wa_s.p,
                                                                            e->auc_wb_s.p, e->auc_pos_of.p, e->auc_price_s.p,
                                                                            use_rep ? e->reputation.p : nullptr, use_rep ? e->auc_rep_s.p : nullptr);
    PM_LAUNCH_CHECK("pm_auction_gather_sorted");
    return PM_OK;
  };
  {
    const int rc = sort_workers();
    if (rc != PM_OK) return rc;
  }
  PM_CUDA(cudaMemsetAsync(e->auc_winner.p, 0xFF, (size_t)std::max<uint32_t>(W, 1) * 4, e->stream));
  // one packed 64-bit sort key per candidate when every reachable cost fits (decided on the device, read by the kernels)
  pm::pm_auction_limits<<<std::max(1u, std::min(blocks_for(std::max(W, T), 256), 592u)), 256, 0, e->stream>>>(e->wb.p, W, e->price_cap.p, T, e->auc_ctl.p);
  pm::pm_auction_decide_packed<<<1, 1, 0, e->stream>>>(e->auc_ctl.p, W, T, e->auc_scale, e->auc_eps_start ? e->auc_eps_start : 1, (uint32_t)e->tune_auction);
  PM_LAUNCH_CHECK("pm_auction_decide_packed");
  PM_CUDA(cudaMemcpyAsync(e->h_ctl.p, e->auc_ctl.p, sizeof(pm::AuctionCtl), cudaMemcpyDeviceToHost, e->stream));
  PM_CUDA(cudaStreamSynchronize(e->stream));
  const bool packed_claim = e->h_ctl.p->packed_claim != 0;   // then no round launches pm_auction_claim at all

  pm::AuctionParams ap;
  ap.ev = eval_params(e);
  ap.wa_s = e->auc_wa_s.p; ap.wb_s = e->auc_wb_s.p; ap.perm = e->auc_perm.p; ap.pos_of = e->auc_pos_of.p; ap.price_s = e->auc_price_s.p;
  ap.csort_s = reinterpret_cast<const unsigned long long*>(e->auc_ckey_s.p);
  ap.rep_s = use_rep ? e->auc_rep_s.p : nullptr; ap.min_rep = use_rep ? e->ask_min_rep.p : nullptr;
  ap.price_cap = e->price_cap.p; ap.price = e->auc_price.p; ap.owner = e->auc_owner.p; ap.assigned = e->auc_assigned.p;
  ap.withdrawn = e->auc_withdrawn.p; ap.active = e->auc_active.p; ap.n_asks = T; ap.bid_w = e->auc_bid_w.p; ap.bid_p = e->auc_bid_p.p;
  ap.bid_max = e->auc_bid_max.p; ap.winner = e->auc_winner.p; ap.scale = (long long)e->auc_scale;
  ap.class_of = e->auc_class_of.p; ap.class_rep = e->auc_class_rep.p; ap.class_req = e->auc_class_req.p;
  ap.cand = e->auc_cand.p; ap.theta = e->auc_theta.p; ap.theta_w = e->auc_theta_w.p;
  ap.pool = e->auc_pool.p; ap.pool_bound_v = e->auc_pool_bound_v.p; ap.pool_bound_w = e->auc_pool_bound_w.p;
  ap.walk_list = e->auc_walk_list.p; ap.split_bound_v = e->auc_split_v.p; ap.split_bound_w = e->auc_split_w.p; ap.split_ticket = e->auc_split_ticket.p; ap.split_first = e->auc_split_first.p;
  ap.skip_key = reinterpret_cast<unsigned long long*>(e->auc_skip_key.p);
  ap.class_list = e->auc_class_list.p; ap.retry = e->auc_retry.p; ap.fallback = e->auc_fallback.p; ap.ctl = e->auc_ctl.p;
  ap.dbg = (uint32_t)e->tune_auction;
  ap.pool_good = e->tune_auc_good > 0 ? (uint32_t)e->tune_auc_good : (uint32_t)pm::kAucPoolGood;
  ap.pool_extra = e->tune_auc_extra > 0 ? (uint32_t)e->tune_auc_extra : (uint32_t)pm::kAucPoolExtra;
  const size_t smem = pm::kAucStages * sizeof(pm::AuctionStage) + sizeof(pm::AuctionMerge);
  PM_CUDA(cudaFuncSetAttribute(pm::pm_auction_scan, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // fixed grids: every kernel strides over a list whose length it reads from the control block
  const unsigned g_scan = kScanGrid;
  const unsigned g_apply = std::max(1u, std::min(blocks_for(T, 256), 148u));   // every CTA pays a fence + the ticket: one per SM at most
  const unsigned g_refill = std::max(1u, std::min(C, 1184u));   // 12 KB of shared memory per CTA: eight per SM
  const unsigned g_warp = std::max(1u, std::min(blocks_for(T, pm::kAucWarps), 1184u));
  const unsigned g_thr = std::max(1u, std::min(blocks_for(T, 256), 592u));
  const uint32_t kBatch = 32;  // rounds launched between polls of the control block
  const uint32_t kResort = (e->tune_auction >> 8) ? (uint32_t)(e->tune_auction >> 8) : 4u;   // batches between re-sorts of the worker copy
  uint64_t eps = e->auc_eps_start ? e->auc_eps_start : 1;
  const uint32_t div = e->auc_eps_div < 2 ? 2 : e->auc_eps_div;
  for (;;) {  // eps phases: assignment cleared, prices (and so the class caches' bounds) kept
    PM_CUDA(cudaMemsetAsync(e->auc_owner.p, 0xFF, (size_t)std::max<uint32_t>(W, 1) * 4, e->stream));
    PM_CUDA(cudaMemsetAsync(e->auc_assigned.p, 0xFF, (size_t)std::max<uint32_t>(T, 1) * 4, e->stream));
    PM_CUDA(cudaMemsetAsync(e->auc_withdrawn.p, 0, (size_t)std::max<uint32_t>(T, 1) * 4, e->stream));
    if (C && eps == (e->auc_eps_start ? e->auc_eps_start : 1)) {  // no cache yet: "invalid" sends every class to a scan
      pm::pm_fill_i64<<<std::min(blocks_for(C, 256), 1184u), 256, 0, e->stream>>>(e->auc_theta.p, pm::kThetaInvalid, C);
      pm::pm_fill_i64<<<std::min(blocks_for(C, 256), 1184u), 256, 0, e->stream>>>(e->auc_pool_bound_v.p, pm::kThetaInvalid, C);
      PM_LAUNCH_CHECK("pm_fill_i64");
    }
    ap.eps = (long long)eps;
    if (T) {
      pm::pm_auction_compact<<<blocks_for(T, 256), 256, 0, e->stream>>>(ap, T);
      PM_LAUNCH_CHECK("pm_auction_compact");
    }
    pm::pm_auction_advance<<<1, 1, 0, e->stream>>>(e->auc_ctl.p, 1);
    PM_LAUNCH_CHECK("pm_auction_advance");
    auto launch_rounds = [&]() {
      for (uint32_t r = 0; r < kBatch; ++r) {
        pm::pm_auction_bid_cached<<<g_warp, pm::kAucThreads, 0, e->stream>>>(ap, 0);
        pm::pm_auction_refill<<<g_refill, pm::kAucThreads, 0, e->stream>>>(ap);
        pm::pm_auction_scan<<<g_scan, pm::kAucThreads, smem, e->stream>>>(ap, 1);
        pm::pm_auction_bid_cached<<<g_warp, pm::kAucThreads, 0, e->stream>>>(ap, 1);
        pm::pm_auction_scan<<<g_scan, pm::kAucThreads, smem, e->stream>>>(ap, 0);
        if (!packed_claim) pm::pm_auction_claim<<<g_thr, 256, 0, e->stream>>>(ap);
        pm::pm_auction_apply<<<g_apply, 256, 0, e->stream>>>(ap);   // ... and the next round's active list, and the advance
      }
    };
    // a batch of rounds is one CUDA graph (the kernels are a few microseconds each: launch-bound otherwise);
    // a stream that cannot be captured (the legacy default stream) gets plain launches
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t graph_exec = nullptr;
    if (T && cudaStreamBeginCapture(e->stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
      launch_rounds();
      if (cudaStreamEndCapture(e->stream, &graph) != cudaSuccess || cudaGraphInstantiate(&graph_exec, graph, 0) != cudaSuccess) {
        if (graph) cudaGraphDestroy(graph);
        graph = nullptr;
        graph_exec = nullptr;
      }
    }
    (void)cudaGetLastError();
    int rc_rounds = PM_OK;
    uint32_t n_batches = 0;
    for (;;) {
      cudaError_t ce = cudaMemcpyAsync(e->h_ctl.p, e->auc_ctl.p, sizeof(pm::AuctionCtl), cudaMemcpyDeviceToHost, e->stream);
      if (ce == cudaSuccess) ce = cudaStreamSynchronize(e->stream);
      if (ce != cudaSuccess) { rc_rounds = e->fail(PM_E_CUDA, std::string("pm_match: auction rounds: ") + cudaGetErrorString(ce)); break; }
      if (e->tune_auction & 4) {   // PM_TUNE_AUCTION=4: one line per batch of rounds
        static thread_local double t_prev = 0;
        timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts);
        const double now = ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
        std::fprintf(stderr, "auction batch: rounds=%u active=%u refills=%llu class_scans=%llu ask_scans=%llu evals=%llu dt_ms=%.2f\n", e->h_ctl.p->rounds,
                     e->h_ctl.p->n_active, e->h_ctl.p->n_refills, e->h_ctl.p->n_class_scans, e->h_ctl.p->n_ask_scans, e->h_ctl.p->evals, t_prev ? now - t_prev : 0.0);
        t_prev = now;
      }
      if (e->h_ctl.p->n_active == 0) break;
      if (e->h_ctl.p->rounds > 50u * 1000u * 1000u) { rc_rounds = e->fail(PM_E_CUDA, "pm_match: auction did not terminate"); break; }
      if (n_batches && n_batches % kResort == 0) {   // bid-up workers move back in the walk order
        const int rc = sort_workers();
        if (rc != PM_OK) { rc_rounds = rc; break; }
      }
      ++n_batches;
      if (graph_exec) ce = cudaGraphLaunch(graph_exec, e->stream);
      else { launch_rounds(); ce = cudaGetLastError(); }
      if (ce != cudaSuccess) { rc_rounds = e->fail(PM_E_CUDA, std::string("pm_match: auction rounds: ") + cudaGetErrorString(ce)); break; }
    }
    if (graph_exec) cudaGraphExecDestroy(graph_exec);
    if (graph) cudaGraphDestroy(graph);
    if (rc_rounds != PM_OK) return rc_rounds;
    if (eps == 1) break;
    eps = std::max<uint64_t>(1, eps / div);
  }
  e->stats.n_rounds = e->h_ctl.p->rounds;
  e->stats.evals = e->h_ctl.p->evals;
  e->stats.n_tiles = (uint32_t)std::min<unsigned long long>(e->h_ctl.p->n_class_scans, 0xFFFFFFFFull);
  e->stats.n_fused_launches = (uint32_t)std::min<unsigned long long>(e->h_ctl.p->n_ask_scans, 0xFFFFFFFFull);
  e->stats.n_launches = e->h_ctl.p->rounds * (packed_claim ? 6u : 7u);
  e->stats.n_build_launches = (uint32_t)std::min<unsigned long long>(e->h_ctl.p->n_refills, 0xFFFFFFFFull);
  tm.stop();
  Timer tr(e, &e->stats.ms_resolve);
  // result: one solo group per assigned ask, ask order
  pm::pm_auction_flags<<<blocks_for((size_t)T + 1, 256), 256, 0, e->stream>>>(e->auc_assigned.p, T, e->auc_flag.p);
  PM_LAUNCH_CHECK("pm_auction_flags");
  {
    size_t tmp = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp, e->auc_flag.p, e->auc_gidx.p, (int)(T + 1), e->stream);
    PM_CUDA(e->cub_tmp.ensure(tmp));
    PM_CUDA(cub::DeviceScan::ExclusiveSum(e->cub_tmp.p, tmp, e->auc_flag.p, e->auc_gidx.p, (int)(T + 1), e->stream));
  }
  PM_CUDA(cudaMemsetAsync(e->worker_group.p, 0xFF, (size_t)std::max<uint32_t>(W, 1) * 4, e->stream));
  PM_CUDA(cudaMemsetAsync(e->worker_ask.p, 0xFF, (size_t)std::max<uint32_t>(W, 1) * 4, e->stream));
  if (T) {
    pm::pm_auction_emit<<<blocks_for(T, 256), 256, 0, e->stream>>>(e->auc_assigned.p, e->auc_gidx.p, e->wb.p, T, e->worker_group.p,
                                                                    e->worker_ask.p, e->group_ask.p, e->group_off.p, e->members.p,
                                                                    e->ask_best.p, e->ask_count.p);
    PM_LAUNCH_CHECK("pm_auction_emit");
  }
  PM_CUDA(cudaMemcpyAsync(e->h_scalars.p + 17, e->auc_gidx.p + T, 4, cudaMemcpyDeviceToHost, e->stream));
  PM_CUDA(cudaStreamSynchronize(e->stream));
  const uint32_t G = e->h_scalars.p[17];
  PM_CUDA(cudaMemcpyAsync(e->group_off.p + G, e->h_scalars.p + 17, 4, cudaMemcpyHostToDevice, e->stream));
  tr.stop();
  e->n_groups = G;
  e->n_assigned = G;
  if (e->cfg.flags & PM_CFG_TIMING) {
    PM_CUDA(cudaEventRecord(e->ev1, e->stream));
    PM_CUDA(cudaEventSynchronize(e->ev1));
    PM_CUDA(cudaEventElapsedTime(&e->stats.ms_total, e->ev0, e->ev1));
    e->resolve_timers();
  }
  e->matched = true;
  e->local_done = false;
  return PM_OK;
}

int pm_set_ask_price_caps(pm_engine* e, const uint32_t* price_cap, uint32_t n_asks) try {
  if (!e) return PM_E_INVALID;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->have_asks || n_asks != e->n_asks) return e->fail(PM_E_INVALID, "pm_set_ask_price_caps: one cap per ask, after pm_set_asks");
  PM_CUDA(cudaSetDevice(e->device));
  PM_CUDA(e->price_cap.ensure(n_asks));
  if (n_asks) PM_CUDA(cudaMemcpyAsync(e->price_cap.p, price_cap, (size_t)n_asks * 4, cudaMemcpyHostToDevice, e->stream));
  PM_CUDA(cudaStreamSynchronize(e->stream));
  e->have_caps = true;
  return PM_OK;
} catch (...) { return pm_guard_rc(); }

// `reputation` worker column and the per-ask floor on it (north-star extension; PM_MODE_AUCTION only)
int pm_set_worker_reputation(pm_engine* e, const uint32_t* reputation, uint32_t first, uint32_t n) try {
  if (!e) return PM_E_INVALID;
  std::lock_guard<std::mutex> lk(e->mu);
  ++e->table_version;
  if (!e->have_workers) return e->fail(PM_E_STATE, "pm_set_worker_reputation: no worker table");
  if ((uint64_t)first + n > e->n_workers) return e->fail(PM_E_INVALID, "pm_set_worker_reputation: range");
  if (n && !reputation) return e->fail(PM_E_INVALID, "pm_set_worker_reputation: null");
  PM_CUDA(cudaSetDevice(e->device));
  if (!e->have_rep) {
    PM_CUDA(e->reputation.ensure(std::max<size_t>(e->wa.n, 1)));
    PM_CUDA(cudaMemsetAsync(e->reputation.p, 0, std::max<size_t>(e->wa.n, 1) * 4, e->stream));
  }
  if (n) PM_CUDA(cudaMemcpyAsync(e->reputation.p + first, reputation, (size_t)n * 4, cudaMemcpyHostToDevice, e->stream));
  PM_CUDA(cudaStreamSynchronize(e->stream));
  e->have_rep = true;
  e->matched = e->local_done = false;
  return PM_OK;
} catch (...) { return pm_guard_rc(); }

int pm_set_ask_min_reputation(pm_engine* e, const uint32_t* min_reputation, uint32_t n_asks) try {
  if (!e) return PM_E_INVALID;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->have_asks || n_asks != e->n_asks) return e->fail(PM_E_INVALID, "pm_set_ask_min_reputation: one floor per ask, after pm_set_asks");
  if (n_asks && !min_reputation) return e->fail(PM_E_INVALID, "pm_set_ask_min_reputation: null");
  PM_CUDA(cudaSetDevice(e->device));
  PM_CUDA(e->ask_min_rep.ensure(std::max<uint32_t>(n_asks, 1)));
  if (n_asks) PM_CUDA(cudaMemcpyAsync(e->ask_min_rep.p, min_reputation, (size_t)n_asks * 4, cudaMemcpyHostToDevice, e->stream));
  PM_CUDA(cudaStreamSynchronize(e->stream));
  e->have_min_rep = true;
  e->auc_classes_valid = false;   // the floor is part of an ask's class
  e->matched = e->local_done = false;
  return PM_OK;
} catch (...) { return pm_guard_rc(); }

int pm_set_auction_params(pm_engine* e, uint64_t cost_scale, uint64_t eps_start, uint32_t eps_div) try {
  if (!e) return PM_E_INVALID;
  std::lock_guard<std::mutex> lk(e->mu);
  e->auc_scale = cost_scale ? cost_scale : 1;
  e->auc_eps_start = eps_start ? eps_start : 1;
  e->auc_eps_div = eps_div < 2 ? 2 : eps_div;
  return PM_OK;
} catch (...) { return pm_guard_rc(); }

// The one data-path exchange of a sharded pass (SURVEY 8e): every rank packs {per-ask (min cost, argmin) and feasible
// count over its workers, first feasible ask of its own workers} into one buffer, ONE all-gather over NVLink moves
// them, and every rank folds the contributions into the same global arrays.  Enqueued on the engine's stream: no host
// synchronisation, nothing but NCCL's kernel between the evaluation and the resolution sweep.
static int exchange_locked(pm_engine* e) {
  const NcclApi& nccl = nccl_api();
  if (!nccl.ok) return e->fail(PM_E_UNSUPPORTED, nccl.err);
  const uint32_t W = e->n_workers, T = e->n_asks, n = e->comm->n_ranks;
  uint32_t w0 = 0, nw = 0;
  e->shard(&w0, &nw);
  const uint32_t per = (uint32_t)(((uint64_t)W + n - 1) / n);
  const size_t stride = (((size_t)T * 12 + (size_t)per * 4) + 15) & ~(size_t)15;
  PM_CUDA(e->xchg_send.ensure(stride));
  PM_CUDA(e->xchg_recv.ensure(stride * n));
  Timer tm(e, &e->stats.ms_exchange);
  const size_t work = std::max<size_t>(std::max<size_t>(T, W), 1);
  pm::pm_xchg_pack<<<std::min(blocks_for(work, 256), 1184u), 256, 0, e->stream>>>(e->first_ask.p + w0, nw, per, e->ask_best.p, e->ask_count.p, T,
                                                                                  e->xchg_send.p);
  PM_LAUNCH_CHECK("pm_xchg_pack");
  const ncclResult_t nr = nccl.AllGather(e->xchg_send.p, e->xchg_recv.p, stride, ncclUint8, e->comm->nccl, e->stream);
  if (nr != ncclSuccess) return e->fail(PM_E_CUDA, std::string("ncclAllGather: ") + nccl.GetErrorString(nr));
  pm::pm_xchg_unpack<<<std::min(blocks_for(work, 256), 1184u), 256, 0, e->stream>>>(e->xchg_recv.p, n, stride, std::max(per, 1u), W, T, e->first_ask.p,
                                                                                    e->ask_best.p, e->ask_count.p);
  PM_LAUNCH_CHECK("pm_xchg_unpack");
  tm.stop();
  e->stats.exchange_bytes = (uint64_t)stride * n;
  return PM_OK;
}

int pm_match_local(pm_engine* e, uint32_t mode) try {
  if (!e) return PM_E_INVALID;
  std::lock_guard<std::mutex> lk(e->mu);
  if ((mode & 0xFFu) == PM_MODE_AUCTION) return e->fail(PM_E_UNSUPPORTED, "pm_match_local: auction mode is single-GPU (use pm_match)");
  return match_local_locked(e, mode);
} catch (...) { return pm_guard_rc(); }
int pm_match_finish(pm_engine* e, uint32_t mode) try {
  if (!e) return PM_E_INVALID;
  std::lock_guard<std::mutex> lk(e->mu);
  return match_finish_locked(e, mode);
} catch (...) { return pm_guard_rc(); }
int pm_match(pm_engine* e, uint32_t mode) try {
  if (!e) return PM_E_INVALID;
  std::lock_guard<std::mutex> lk(e->mu);
  if ((mode & 0xFFu) == PM_MODE_AUCTION) return match_auction_locked(e);
  int rc = match_local_locked(e, mode);
  if (rc != PM_OK) return rc;
  if (e->comm && e->comm->n_ranks > 1) {
    rc = exchange_locked(e);
    if (rc != PM_OK) return rc;
  }
  return match_finish_locked(e, mode);
} catch (...) { return pm_guard_rc(); }

int pm_set_shard(pm_engine* e, uint32_t first, uint32_t count) try {
  if (!e) return PM_E_INVALID;
  std::lock_guard<std::mutex> lk(e->mu);
  e->cfg.shard_first = first;
  e->cfg.shard_count = count;
  e->matched = e->local_done = false;
  return PM_OK;
} catch (...) { return pm_guard_rc(); }

// ------------------------------------------------------------------ communicators
int pm_comm_unique_id(uint8_t* id_out) try {
  if (!id_out) return PM_E_INVALID;
  const NcclApi& nccl = nccl_api();
  if (!nccl.ok) { g_create_error = nccl.err; return PM_E_UNSUPPORTED; }
  static_assert(sizeof(ncclUniqueId) == PM_COMM_ID_BYTES, "ncclUniqueId size");
  ncclUniqueId id;
  const ncclResult_t nr = nccl.GetUniqueId(&id);
  if (nr != ncclSuccess) { g_create_error = std::string("ncclGetUniqueId: ") + nccl.GetErrorString(nr); return PM_E_CUDA; }
  std::memcpy(id_out, &id, sizeof id);
  return PM_OK;
} catch (...) { return pm_guard_rc(); }

int pm_comm_create(const uint8_t* unique_id, uint32_t n_ranks, uint32_t rank, int32_t device, pm_comm** out) try {
  if (!unique_id || !out || n_ranks == 0 || rank >= n_ranks) return PM_E_INVALID;
  *out = nullptr;
  const NcclApi& nccl = nccl_api();
  if (!nccl.ok) { g_create_error = nccl.err; return PM_E_UNSUPPORTED; }
  if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); g_create_error = "pm_comm_create: bad device"; return PM_E_INVALID; }
  ncclUniqueId id;
  std::memcpy(&id, unique_id, sizeof id);
  pm_comm* c = new pm_comm;
  c->n_ranks = n_ranks; c->rank = rank; c->device = device;
  const ncclResult_t nr = nccl.CommInitRank(&c->nccl, (int)n_ranks, id, (int)rank);
  if (nr != ncclSuccess) {
    g_create_error = std::string("ncclCommInitRank: ") + nccl.GetErrorString(nr);
    delete c;
    return PM_E_CUDA;
  }
  *out = c;
  return PM_OK;
} catch (...) { return pm_guard_rc(); }

void pm_comm_destroy(pm_comm* c) {
  if (!c) return;
  if (c->nccl && nccl_api().ok) {
    cudaSetDevice(c->device);
    nccl_api().CommDestroy(c->nccl);
  }
  delete c;
}

int pm_attach_comm(pm_engine* e, pm_comm* c) try {
  if (!e) return PM_E_INVALID;
  std::lock_guard<std::mutex> lk(e->mu);
  if (c && c->device != e->device) return e->fail(PM_E_INVALID, "pm_attach_comm: communicator and engine are on different devices");
  e->comm = c;
  e->matched = e->local_done = false;
  return PM_OK;
} catch (...) { return pm_guard_rc(); }


int pm_fetch_result(pm_engine* e, pm_result* out) try {
  if (!e || !out) return PM_E_INVALID;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->matched) return e->fail(PM_E_STATE, "pm_fetch_result: no completed match");
  PM_CUDA(cudaSetDevice(e->device));
  const uint32_t W = e->n_workers, T = e->n_asks, G = e->n_groups, M = e->n_assigned;
  PM_CUDA(e->r_worker_group.ensure(W)); PM_CUDA(e->r_worker_ask.ensure(W));
  PM_CUDA(e->r_group_ask.ensure(G)); PM_CUDA(e->r_group_off.ensure((size_t)G + 1));
  PM_CUDA(e->r_members.ensure(M)); PM_CUDA(e->r_ask_best.ensure(T)); PM_CUDA(e->r_ask_count.ensure(T));
  if (W) {
    PM_CUDA(cudaMemcpyAsync(e->r_worker_group.p, e->worker_group.p, (size_t)W * 4, cudaMemcpyDeviceToHost, e->stream));
    PM_CUDA(cudaMemcpyAsync(e->r_worker_ask.p, e->worker_ask.p, (size_t)W * 4, cudaMemcpyDeviceToHost, e->stream));
  }
  if (G) PM_CUDA(cudaMemcpyAsync(e->r_group_ask.p, e->group_ask.p, (size_t)G * 4, cudaMemcpyDeviceToHost, e->stream));
  PM_CUDA(cudaMemcpyAsync(e->r_group_off.p, e->group_off.p, ((size_t)G + 1) * 4, cudaMemcpyDeviceToHost, e->stream));
  if (M) PM_CUDA(cudaMemcpyAsync(e->r_members.p, e->members.p, (size_t)M * 4, cudaMemcpyDeviceToHost, e->stream));
  if (T) {
    PM_CUDA(cudaMemcpyAsync(e->r_ask_best.p, e->ask_best.p, (size_t)T * 8, cudaMemcpyDeviceToHost, e->stream));
    PM_CUDA(cudaMemcpyAsync(e->r_ask_count.p, e->ask_count.p, (size_t)T * 4, cudaMemcpyDeviceToHost, e->stream));
  }
  PM_CUDA(cudaStreamSynchronize(e->stream));
  out->n_workers = W; out->n_asks = T; out->n_groups = G; out->n_members = M;
  out->worker_group = e->r_worker_group.p; out->worker_ask = e->r_worker_ask.p;
  out->group_ask = e->r_group_ask.p; out->group_off = e->r_group_off.p; out->group_members = e->r_members.p;
  out->ask_best = (const int64_t*)e->r_ask_best.p; out->ask_count = e->r_ask_count.p;
  out->stats = e->stats;
  return PM_OK;
} catch (...) { return pm_guard_rc(); }

int pm_build_cost_tile(pm_engine* e, uint32_t t0, uint32_t nt, int64_t* host_out) try {
  if (!e || !host_out) return PM_E_INVALID;
  std::lock_guard<std::mutex> lk(e->mu);
  if (!e->have_workers || !e->have_asks) return e->fail(PM_E_STATE, "pm_build_cost_tile: tables not set");
  if (e->max_pattern_row > e->n_patterns || (e->max_pattern_row && !e->have_bits))
    return e->fail(PM_E_STATE, "pm_build_cost_tile: model table missing");
  if ((uint64_t)t0 + nt > e->n_asks || nt == 0) return e->fail(PM_E_INVALID, "pm_build_cost_tile: ask range");
  PM_CUDA(cudaSetDevice(e->device));
  const uint32_t W = e->n_workers;
  uint32_t w0 = 0, nw = 0;
  e->shard(&w0, &nw);
  if (nw == 0 || (uint64_t)w0 + nw > W) return e->fail(PM_E_INVALID, "pm_build_cost_tile: empty worker range");
  if (!e->have_bits) {
    PM_CUDA(e->bits.ensure(1));
    PM_CUDA(cudaMemsetAsync(e->bits.p, 0xFF, 4, e->stream));
    e->words = 1;
  }
  const size_t ld = (((size_t)nw + pm::kEvalCols - 1) / pm::kEvalCols) * pm::kEvalCols;
  if (nt > 65535u * pm::kEvalRows) return e->fail(PM_E_INVALID, "pm_build_cost_tile: too many rows");
  pm::EvalParams p = eval_params(e);
  dim3 grid(blocks_for(ld, pm::kEvalCols), blocks_for(nt, pm::kEvalRows));
  bool fast = false;
  int bits_mode = ((uint64_t)p.n_bits_rows * p.words <= (uint64_t)pm::kBitsCap) ? (p.words == 1 ? 2 : 1) : 0;
  {
    int rc = decide_fast(e, &fast);
    if (rc != PM_OK) return rc;
    const bool wm = fast && bits_mode == 0 && p.n_bits_rows <= 31u && e->tune_build != 7;   // as pm_match
    if (wm) {
      rc = worker_major(e, &p, &bits_mode);
      if (rc != PM_OK) return rc;
    }
    rc = bind_rows(e, wm);
    if (rc != PM_OK) return rc;
  }
  // the kernel pm_match would run: with 16-bit words the tile goes after the int64 one and is widened into it
  const bool narrow = narrow_cost(e, fast, bits_mode);
  const size_t wide_bytes = (size_t)nt * ld * 8;
  if (e->cost.ensure(wide_bytes + (narrow ? (size_t)nt * ld * 2 : 0)) != cudaSuccess) {
    cudaGetLastError();
    return e->fail(PM_E_NOMEM, "pm_build_cost_tile: cannot allocate the tile");
  }
  if (narrow) {
    launch_build(e, p, bits_mode, fast, true, grid, t0, nt, w0, nw, ld, e->cost.p + wide_bytes);
    PM_LAUNCH_CHECK("pm_build_cost");
    pm::pm_widen_cost<<<std::min(blocks_for((size_t)nt * ld, 256), 4096u), 256, 0, e->stream>>>(
        reinterpret_cast<const uint16_t*>(e->cost.p + wide_bytes), (size_t)nt * ld, ld, w0, reinterpret_cast<long long*>(e->cost.p));
    PM_LAUNCH_CHECK("pm_widen_cost");
  } else {
    launch_build(e, p, bits_mode, fast, false, grid, t0, nt, w0, nw, ld, e->cost.p);
    PM_LAUNCH_CHECK("pm_build_cost");
  }
  PM_CUDA(cudaMemcpy2DAsync(host_out, (size_t)nw * 8, e->cost.p, ld * 8, (size_t)nw * 8, nt,
                            cudaMemcpyDeviceToHost, e->stream));
  PM_CUDA(cudaStreamSynchronize(e->stream));
  return PM_OK;
} catch (...) { return pm_guard_rc(); }

int pm_get_stats(const pm_engine* e, pm_stats* out) try {
  if (!e || !out) return PM_E_INVALID;
  *out = e->stats;
  return PM_OK;
} catch (...) { return pm_guard_rc(); }

int pm_device_buffer(pm_engine* e, uint32_t which, void** dev_ptr, size_t* bytes) try {
  if (!e || !dev_ptr || !bytes) return PM_E_INVALID;
  std::lock_guard<std::mutex> lk(e->mu);
  switch (which) {
    case PM_BUF_WORKER_FIRST_ASK: *dev_ptr = e->first_ask.p; *bytes = (size_t)e->n_workers * 4; break;
    case PM_BUF_ASK_BEST: *dev_ptr = e->ask_best.p; *bytes = (size_t)e->n_asks * 8; break;
    case PM_BUF_ASK_COUNT: *dev_ptr = e->ask_count.p; *bytes = (size_t)e->n_asks * 4; break;
    default: return e->fail(PM_E_INVALID, "pm_device_buffer: unknown buffer");
  }
  if (!*dev_ptr) return e->fail(PM_E_STATE, "pm_device_buffer: buffer not allocated yet (run pm_match_local)");
  return PM_OK;
} catch (...) { return pm_guard_rc(); }

int pm_stream_sync(pm_engine* e) try {
  if (!e) return PM_E_INVALID;
  PM_CUDA(cudaSetDevice(e->device));
  PM_CUDA(cudaStreamSynchronize(e->stream));
  return PM_OK;
} catch (...) { return pm_guard_rc(); }

// ------------------------------------------------------------------ one process, several GPUs
// The orchestrator is one process with one management loop (reference crates/orchestrator/src/main.rs:283-289), so
// the multi-GPU form it can call is this one: N engines, one per device, each with the full (small) tables and an
// equal share of the canonical worker order; communicators from ncclCommInitAll; a pass = every device evaluates its
// share, one all-gather, every device runs the same resolution sweep (engine 0's result is the result).
struct pm_multi {
  std::vector<pm_engine*> engines;
  std::vector<pm_comm*> comms;
  std::string err;
};

void pm_multi_destroy(pm_multi* m) {
  if (!m) return;
  for (pm_engine* e : m->engines) pm_destroy(e);
  for (pm_comm* c : m->comms) pm_comm_destroy(c);
  delete m;
}

int pm_multi_create(const pm_cfg* cfg, const int32_t* devices, uint32_t n, pm_multi** out) try {
  if (!cfg || !devices || !out || n == 0) return PM_E_INVALID;
  *out = nullptr;
  pm_multi* m = new pm_multi;
  for (uint32_t i = 0; i < n; ++i) {
    pm_cfg c = *cfg;
    c.device = devices[i];
    c.shard_first = c.shard_count = 0;
    c.stream = nullptr;   // one private stream per device
    pm_engine* e = nullptr;
    const int rc = pm_create(&c, &e);
    if (rc != PM_OK) { pm_multi_destroy(m); return rc; }
    m->engines.push_back(e);
  }
  if (n > 1) {
    const NcclApi& nccl = nccl_api();
    if (!nccl.ok) { g_create_error = nccl.err; pm_multi_destroy(m); return PM_E_UNSUPPORTED; }
    std::vector<ncclComm_t> raw(n, nullptr);
    std::vector<int> devs(devices, devices + n);
    const ncclResult_t nr = nccl.CommInitAll(raw.data(), (int)n, devs.data());
    if (nr != ncclSuccess) {
      g_create_error = std::string("ncclCommInitAll: ") + nccl.GetErrorString(nr);
      pm_multi_destroy(m);
      return PM_E_CUDA;
    }
    for (uint32_t i = 0; i < n; ++i) {
      pm_comm* c = new pm_comm;
      c->nccl = raw[i]; c->n_ranks = n; c->rank = i; c->device = devices[i];
      m->comms.push_back(c);
      m->engines[i]->comm = c;
    }
  }
  *out = m;
  return PM_OK;
} catch (...) { return pm_guard_rc(); }

uint32_t pm_multi_size(const pm_multi* m) { return m ? (uint32_t)m->engines.size() : 0u; }
pm_engine* pm_multi_engine(pm_multi* m, uint32_t i) { return (m && i < m->engines.size()) ? m->engines[i] : nullptr; }
const char* pm_multi_last_error(const pm_multi* m) { return m ? m->err.c_str() : g_create_error.c_str(); }

#define PM_MULTI_EACH(call)                                      \
  do {                                                           \
    if (!m) return PM_E_INVALID;                                 \
    for (pm_engine* e : m->engines) {                            \
      const int rc_ = (call);                                    \
      if (rc_ != PM_OK) { m->err = pm_last_error(e); return rc_; } \
    }                                                            \
    return PM_OK;                                                \
  } while (0)

int pm_multi_set_asks(pm_multi* m, const pm_ask* asks, uint32_t n_asks, const pm_gpu_opt* opts, uint32_t n_opts) try {
  PM_MULTI_EACH(pm_set_asks(e, asks, n_asks, opts, n_opts));
} catch (...) { return pm_guard_rc(); }
int pm_multi_set_model_table(pm_multi* m, const uint32_t* bits, uint32_t n_patterns, uint32_t n_models, uint32_t words) try {
  PM_MULTI_EACH(pm_set_model_table(e, bits, n_patterns, n_models, words));
} catch (...) { return pm_guard_rc(); }
int pm_multi_set_worker_count(pm_multi* m, uint32_t n_workers) try {
  PM_MULTI_EACH(pm_set_worker_count(e, n_workers));
} catch (...) { return pm_guard_rc(); }
int pm_multi_upsert_workers(pm_multi* m, const pm_worker_a* a, const pm_worker_b* b, uint32_t first, uint32_t n) try {
  PM_MULTI_EACH(pm_upsert_workers(e, a, b, first, n));
} catch (...) { return pm_guard_rc(); }
int pm_multi_set_worker_locations(pm_multi* m, const double* lat, const double* lon, uint32_t first, uint32_t n) try {
  PM_MULTI_EACH(pm_set_worker_locations(e, lat, lon, first, n));
} catch (...) { return pm_guard_rc(); }
int pm_multi_set_worker_addr_rank(pm_multi* m, const uint32_t* rank, uint32_t first, uint32_t n) try {
  PM_MULTI_EACH(pm_set_worker_addr_rank(e, rank, first, n));
} catch (...) { return pm_guard_rc(); }
int pm_multi_set_flags(pm_multi* m, const uint32_t* idx, const uint32_t* flags, uint32_t n) try {
  PM_MULTI_EACH(pm_set_flags(e, idx, flags, n));
} catch (...) { return pm_guard_rc(); }
int pm_multi_sync(pm_multi* m) try {
  PM_MULTI_EACH(pm_stream_sync(e));
} catch (...) { return pm_guard_rc(); }
#undef PM_MULTI_EACH

int pm_multi_match(pm_multi* m, uint32_t mode) try {
  if (!m) return PM_E_INVALID;
  const size_t n = m->engines.size();
  if (n == 1) {
    const int rc = pm_match(m->engines[0], mode);
    if (rc != PM_OK) m->err = pm_last_error(m->engines[0]);
    return rc;
  }
  // a rank that fails before the collective would leave the others waiting in it: check what can be checked first,
  // and abort every communicator if a rank still fails on the way
  for (pm_engine* e : m->engines) {
    if (!e->have_workers || !e->have_asks) { m->err = "pm_multi_match: worker and ask tables must be set first"; return PM_E_STATE; }
    if (e->n_workers != m->engines[0]->n_workers || e->n_asks != m->engines[0]->n_asks) {
      m->err = "pm_multi_match: engines hold different tables";
      return PM_E_STATE;
    }
  }
  std::vector<int> rcs(n, PM_OK);
  std::atomic<bool> aborted{false};
  std::vector<std::thread> threads;
  for (size_t i = 0; i < n; ++i) {
    threads.emplace_back([&, i] {
      rcs[i] = pm_match(m->engines[i], mode);
      if (rcs[i] != PM_OK && !aborted.exchange(true) && nccl_api().ok)
        for (pm_comm* c : m->comms)
          if (c->nccl) { nccl_api().CommAbort(c->nccl); c->nccl = nullptr; }
    });
  }
  for (auto& t : threads) t.join();
  for (size_t i = 0; i < n; ++i)
    if (rcs[i] != PM_OK) { m->err = pm_last_error(m->engines[i]); return rcs[i]; }
  return PM_OK;
} catch (...) { return pm_guard_rc(); }

int pm_multi_fetch_result(pm_multi* m, pm_result* out) try {
  if (!m || m->engines.empty()) return PM_E_INVALID;
  const int rc = pm_fetch_result(m->engines[0], out);
  if (rc != PM_OK) m->err = pm_last_error(m->engines[0]);
  return rc;
} catch (...) { return pm_guard_rc(); }

}  // extern "C"
