// skyopt.cu -- host side of libskyopt: catalog upload, workspace management
// and the C-ABI entry points declared in include/skyopt.h.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo
//        -fmad=false -shared -Xcompiler -fPIC  (see __graft_entry__.build()).
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <unordered_map>
#include <array>
#include <vector>

#include "skyopt.h"
#include "skyopt_kernels.cuh"
#include "skyopt_fast.cuh"
#include "skyopt_step.cuh"

using namespace skyopt;

namespace {

thread_local std::string g_error;

int fail(int code, const char *fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_error = buf;
  return code;
}

#define CU(expr)                                                            \
  do {                                                                      \
    cudaError_t e_ = (expr);                                                \
    if (e_ != cudaSuccess)                                                  \
      return fail(SKYOPT_ECUDA, "%s failed: %s (%s:%d)", #expr,             \
                  cudaGetErrorString(e_), __FILE__, __LINE__);              \
  } while (0)

// NVTX range around a native entry point (shows up in Nsight timelines next
// to the host events of skypilot_b200/utils/timeline.py).
struct NvtxRange {
  explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }
inline int next_pow2(int x) { int p = 1; while (p < x) p <<= 1; return p; }

// Private stream + buffers of one in-flight call.
struct Ctx {
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[8] = {};
  char *dbuf = nullptr; size_t dcap = 0;   // device workspace
  char *hbuf = nullptr; size_t hcap = 0;   // pinned staging
  uint32_t *flush = nullptr; size_t flush_words = 0;
  unsigned long long *trace = nullptr;  // SKYOPT_TRACE: device-side timeline
  unsigned int *sync = nullptr;         // step_kernel's barrier counter: monotone, never reset in a launch
  unsigned int sync_total = 0;          // arrivals expected so far (the next launch's barrier target)
};

// Bump allocator over one buffer; first pass (base == nullptr) only sizes.
struct Carver {
  char *base; size_t off = 0;
  explicit Carver(char *b) : base(b) {}
  template <typename T> T *take(size_t n) {
    off = align_up(off);
    T *p = base ? reinterpret_cast<T *>(base + off) : nullptr;
    off += n * sizeof(T);
    return p;
  }
};

}  // namespace

struct SkyoptCatalog {
  int device = 0;
  CatDev dev{};
  // flag_density[c][m]: fraction of cloud c's 128-row chunks whose summary
  // carries every flag bit of m -- how often a query requiring m survives the
  // zone-map test (used to size the scan's query groups).
  std::vector<std::array<float, 256>> flag_density;
  // Static tile classes. For every tile size (256 << r rows, r = 0..2) the
  // tiles of a cloud are split into those where default-family rows are
  // common ("dense": requests without accelerators match most of their rows)
  // and the rest; each class has its own flag_density, so the dense part of a
  // catalog can be scanned with few queries per block and the sparse part
  // with all of them fused.
  struct TileClass {
    int n_tiles = 0;
    int list0 = -1;  // offset into the device tile list; -1 = the run of
    int tile0 = 0;   //   n_tiles consecutive tiles starting at tile0
    std::array<float, 256> density{};
  };
  std::vector<std::array<TileClass, 2>> tile_class[3];  // [r][cloud][0 sparse, 1 dense]
  const int32_t *d_tile_list = nullptr;
  std::vector<void *> allocs;
  int64_t device_bytes = 0;
  std::vector<int32_t> cloud_row_offsets, cloud_inst_offsets, cloud_n_zones,
      cloud_region_offsets;
  std::vector<int32_t> cloud_group_cap;  // max rows of one expand group
  int sort_n = 2, max_regions = 1, max_zones = 1;
  int sm_count = 148;
  int scan_mode = 0;  // 0 auto, 1 one tile per block, 2 streaming (TMA) kernel
  // round-2 fast path (skyopt_fast.cuh): rank / class layouts and static
  // launchable orders; fast_ok = the class dictionaries fit shared memory
  FastCat fast{};
  bool fast_ok = false;
  bool noprune = false;   // stress mode: scan2 ignores the zone map and the bound
  bool split = false;     // fast path as separate launches (scan2, place, solve) instead of step_kernel
  bool coop = false;      // device supports cooperative launches
  std::vector<int32_t> n_cm, n_fa, n_rz;   // class counts per cloud
  std::vector<int32_t> cm_off, fa_off, rz_off;  // [n_clouds + 1] into the dictionaries
  int64_t fast_bytes = 0;
  std::mutex mu;
  std::vector<Ctx *> free_ctx;
};

namespace {

template <typename T>
int upload(SkyoptCatalog *c, const T *src, size_t n, size_t slack, const T **dst,
           int fill = 0) {
  T *p = nullptr;
  const size_t bytes = (n + slack) * sizeof(T);
  CU(cudaMalloc(&p, std::max<size_t>(bytes, 256)));
  c->allocs.push_back(p);
  c->device_bytes += bytes;
  CU(cudaMemset(p, fill, std::max<size_t>(bytes, 256)));
  if (n && src) CU(cudaMemcpy(p, src, n * sizeof(T), cudaMemcpyHostToDevice));
  *dst = p;
  return 0;
}

#include "skyopt_fast_host.inc"

int acquire(SkyoptCatalog *c, Ctx **out) {
  {
    std::lock_guard<std::mutex> g(c->mu);
    if (!c->free_ctx.empty()) {
      *out = c->free_ctx.back();
      c->free_ctx.pop_back();
      return 0;
    }
  }
  Ctx *x = new (std::nothrow) Ctx();
  if (!x) return fail(SKYOPT_ENOMEM, "out of host memory");
  CU(cudaStreamCreateWithFlags(&x->stream, cudaStreamNonBlocking));
  for (auto &e : x->ev) CU(cudaEventCreate(&e));
  CU(cudaMalloc(&x->sync, 256));
  CU(cudaMemset(x->sync, 0, 256));
  *out = x;
  return 0;
}

void release(SkyoptCatalog *c, Ctx *x) {
  std::lock_guard<std::mutex> g(c->mu);
  c->free_ctx.push_back(x);
}

int ensure(Ctx *x, size_t dbytes, size_t hbytes) {
  if (dbytes > x->dcap) {
    if (x->dbuf) CU(cudaFree(x->dbuf));
    x->dbuf = nullptr; x->dcap = 0;
    const size_t cap = align_up(dbytes + dbytes / 4, 1 << 20);
    CU(cudaMalloc(&x->dbuf, cap));
    // result fields a kernel does not write for a given problem (e.g. the
    // chosen candidate of a DAG without a plan) are copied back as zeros
    CU(cudaMemset(x->dbuf, 0, cap));
    x->dcap = cap;
  }
  if (hbytes > x->hcap) {
    if (x->hbuf) CU(cudaFreeHost(x->hbuf));
    x->hbuf = nullptr; x->hcap = 0;
    const size_t cap = align_up(hbytes + hbytes / 4, 1 << 16);
    CU(cudaMallocHost(&x->hbuf, cap));
    x->hcap = cap;
  }
  return 0;
}

// Everything one call needs, laid out twice (host staging / device).
struct Plan {
  // sizes
  int nq = 0, nsets = 0, ns = 0, nt = 0, np = 0, ntar = 0, nb = 0, nd = 0, nres = 0;
  int n_groups = 0, n_blocks = 0, rpt = 4, tpb = 1, nsq = 0; bool stream = false; bool queue = false; bool want_finalize = true;
  int64_t n_partials = 0, list_entries = 0, fuzzy_entries = 0;
  int64_t cand_cap = 0;   // expand candidate buffers
  int64_t scan_rows = 0, pass_rows = 0;
  // round-2 fast path (scan2_kernel + place_kernel)
  bool fast = false; mutable bool fresh_inputs = true; mutable int parity = 0; int n_groups2 = 0, n_pieces = 0, scan2_grid = 0, smem_fa = 0, smem_cm = 0;
  size_t scan2_smem = 0; int64_t layout_rows = 0;
  Scan2Group *groups2; const Scan2Group *host_groups2 = nullptr; uint32_t *best_rank, *any_in;
  PlaceTask *ptasks; SlotAux *saux; uint32_t cap_fa = 0, cap_cm = 0, cap_rz = 0;
  int32_t *dag_done; TaskMin *task_mv; uint32_t *shared_tables; unsigned int *group_ready; bool chain_dags = false; int step_grid = 0; size_t step_smem = 0; mutable bool ran_fused = false;
  // input region (mirrored host/device)
  size_t in_bytes = 0;
  SkyoptQuery *queries; uint32_t *acc_sets; SkyoptSlot *slots; SkyoptTask *tasks;
  int32_t *parents; double *tariffs; SkyoptBlocked *blocked; SkyoptDag *dags;
  SkyoptReservation *res;
  ScanQuery *squeries; QueryTest *qtests; ScanGroup *groups; const ScanGroup *host_groups = nullptr; int32_t *partial_base, *partial_count;
  int64_t *list_base, *fuzzy_base, *slot_off, *task_off; int32_t *task_dag;
  // device-only scratch
  ScanPartial *partials; unsigned long long *list_min, *fuzzy_min, *gbest;
  int32_t *cand_region, *cand_zone; double *cand_pa, *cand_pb;
  int32_t *tc_ref, *tc_slot, *tc_cloud; double *tc_hourly, *tc_value, *dp;
  int32_t *back; int32_t *err_flag;
  // output region (device, copied back in one piece)
  size_t out_off = 0, out_bytes = 0;
  ScanFinal *finals; uint32_t *any1; int32_t *slot_count, *slot_inst;
  SkyoptCandidate *chosen; int32_t *chosen_index, *task_n; SkyoptDagResult *dagres;
  int32_t *err_out;
  size_t total_bytes = 0;
};

void carve_inputs(Plan &P, Carver &c) {
  P.queries = c.take<SkyoptQuery>(P.nq);
  P.acc_sets = c.take<uint32_t>((size_t)P.nsets * SKYOPT_ACC_SET_WORDS);
  P.slots = c.take<SkyoptSlot>(P.ns);
  P.tasks = c.take<SkyoptTask>(P.nt);
  P.parents = c.take<int32_t>(P.np);
  P.tariffs = c.take<double>(P.ntar);
  P.blocked = c.take<SkyoptBlocked>(P.nb);
  P.dags = c.take<SkyoptDag>(P.nd);
  P.res = c.take<SkyoptReservation>(P.nres);
  P.squeries = c.take<ScanQuery>(P.nsq);
  P.qtests = c.take<QueryTest>(P.nsq);
  P.groups = c.take<ScanGroup>(P.n_groups);
  P.partial_base = c.take<int32_t>(P.nq);
  P.partial_count = c.take<int32_t>(P.nq);
  P.list_base = c.take<int64_t>(P.nq);
  P.fuzzy_base = c.take<int64_t>(P.nq);
  P.slot_off = c.take<int64_t>(P.ns);
  P.task_off = c.take<int64_t>(P.nt + 1);
  P.task_dag = c.take<int32_t>(P.nt);
  P.groups2 = c.take<Scan2Group>(P.n_groups2);
  P.ptasks = c.take<PlaceTask>(P.fast ? P.nt : 0);
  P.saux = c.take<SlotAux>(P.fast ? P.ns : 0);
  P.dag_done = c.take<int32_t>(P.fast ? P.nd : 0);
  // two copies: a launch works on one and re-arms the other for the next
  // launch of a device-resident loop (skyopt_optimize_timed), off its own path
  P.group_ready = c.take<unsigned int>(2 * (size_t)P.n_groups2);
  P.best_rank = c.take<uint32_t>(P.fast ? 2 * (size_t)P.nq : 0);
  P.any_in = c.take<uint32_t>(P.fast ? 2 * (size_t)P.nq : 0);
}

void carve_rest(Plan &P, Carver &c) {
  P.partials = c.take<ScanPartial>(P.n_partials);
  P.list_min = c.take<unsigned long long>(P.list_entries);
  P.fuzzy_min = c.take<unsigned long long>(P.fuzzy_entries);
  P.gbest = c.take<unsigned long long>(P.nsq);
  P.task_mv = c.take<TaskMin>(P.fast ? (size_t)P.nt * SKYOPT_MAX_CLOUDS : 0);
  P.shared_tables = c.take<uint32_t>((size_t)P.n_groups2 * (2 * P.cap_fa + P.cap_cm + P.cap_rz));
  P.cand_region = c.take<int32_t>(P.cand_cap);
  P.cand_zone = c.take<int32_t>(P.cand_cap);
  P.cand_pa = c.take<double>(P.cand_cap);
  P.cand_pb = c.take<double>(P.cand_cap);
  P.tc_ref = c.take<int32_t>(P.cand_cap);
  P.tc_slot = c.take<int32_t>(P.cand_cap);
  P.tc_cloud = c.take<int32_t>(P.cand_cap);
  P.tc_hourly = c.take<double>(P.cand_cap);
  P.tc_value = c.take<double>(P.cand_cap);
  P.dp = c.take<double>(P.cand_cap);
  P.back = c.take<int32_t>(P.cand_cap);
  P.err_flag = c.take<int32_t>(1);
  c.off = align_up(c.off);
  P.out_off = c.off;
  P.finals = c.take<ScanFinal>(P.nq);
  P.any1 = c.take<uint32_t>(P.nq);
  P.slot_count = c.take<int32_t>(P.ns);
  P.slot_inst = c.take<int32_t>(P.ns);
  P.chosen = c.take<SkyoptCandidate>(P.nt);
  P.chosen_index = c.take<int32_t>(P.nt);
  P.task_n = c.take<int32_t>(P.nt);
  P.dagres = c.take<SkyoptDagResult>(P.nd);
  P.err_out = c.take<int32_t>(1);
  c.off = align_up(c.off);
  P.out_bytes = c.off - P.out_off;
}

int validate_problem(const SkyoptCatalog *cat, const SkyoptProblem *pb) {
  const int C = cat->dev.n_clouds;
  for (int i = 0; i < pb->n_queries; ++i) {
    const SkyoptQuery &q = pb->queries[i];
    if (q.cloud < 0 || q.cloud >= C) return fail(SKYOPT_EINVAL, "query %d: bad cloud %d", i, q.cloud);
    if (q.acc_set >= pb->n_acc_sets || q.fuzzy_set >= pb->n_acc_sets)
      return fail(SKYOPT_EINVAL, "query %d: accelerator set out of range", i);
    if ((q.qflags & SKYOPT_Q_ACC) && q.acc_set < 0)
      return fail(SKYOPT_EINVAL, "query %d: accelerator query without a set", i);
    if (q.price_col != 0 && q.price_col != 1) return fail(SKYOPT_EINVAL, "query %d: bad price_col", i);
  }
  for (int i = 0; i < pb->n_slots; ++i) {
    const SkyoptSlot &s = pb->slots[i];
    if (s.cloud < 0 || s.cloud >= C) return fail(SKYOPT_EINVAL, "slot %d: bad cloud", i);
    if (s.query >= pb->n_queries || s.gate_query >= pb->n_queries)
      return fail(SKYOPT_EINVAL, "slot %d: query out of range", i);
    if (s.query < 0 && s.inst_id < -2) return fail(SKYOPT_EINVAL, "slot %d: no instance type", i);
    if (s.inst_id >= cat->dev.n_inst) return fail(SKYOPT_EINVAL, "slot %d: instance id out of range", i);
    if (s.acc_set >= pb->n_acc_sets) return fail(SKYOPT_EINVAL, "slot %d: accelerator set out of range", i);
    if (s.region_set >= pb->n_acc_sets) return fail(SKYOPT_EINVAL, "slot %d: region set out of range", i);
    if (s.query < 0 && s.inst_id == -1) return fail(SKYOPT_EINVAL, "slot %d: neither query nor instance", i);
  }
  for (int i = 0; i < pb->n_tasks; ++i) {
    const SkyoptTask &t = pb->tasks[i];
    if (t.slot_begin < 0 || t.slot_end < t.slot_begin || t.slot_end > pb->n_slots)
      return fail(SKYOPT_EINVAL, "task %d: bad slot range", i);
    if (t.n_parents < 0 || t.parent_begin < 0 || t.parent_begin + t.n_parents > pb->n_parents)
      return fail(SKYOPT_EINVAL, "task %d: bad parent range", i);
    if (t.n_parents > 0 && (t.edge_tariff_begin < 0 ||
                            t.edge_tariff_begin + t.n_parents * C > pb->n_tariffs))
      return fail(SKYOPT_EINVAL, "task %d: bad tariff range", i);
    if (t.src_tariff_begin >= 0 && t.src_tariff_begin + C > pb->n_tariffs)
      return fail(SKYOPT_EINVAL, "task %d: bad source tariff range", i);
  }
  for (int i = 0; i < pb->n_dags; ++i) {
    const SkyoptDag &d = pb->dags[i];
    if (d.task_begin < 0 || d.task_end <= d.task_begin || d.task_end > pb->n_tasks)
      return fail(SKYOPT_EINVAL, "dag %d: bad task range", i);
    if (d.blocked_begin < 0 || d.blocked_end < d.blocked_begin || d.blocked_end > pb->n_blocked)
      return fail(SKYOPT_EINVAL, "dag %d: bad blocked range", i);
    for (int t = d.task_begin; t < d.task_end; ++t) {
      const SkyoptTask &tk = pb->tasks[t];
      for (int k = 0; k < tk.n_parents; ++k) {
        const int lp = pb->parents[tk.parent_begin + k];
        if (lp < 0 || lp >= t - d.task_begin)
          return fail(SKYOPT_EINVAL, "dag %d: task order is not topological", i);
      }
      if (d.is_chain && tk.n_parents != (t == d.task_begin ? 0 : 1))
        return fail(SKYOPT_EINVAL, "dag %d: not a chain", i);
      if (d.is_chain && tk.n_parents == 1 && pb->parents[tk.parent_begin] != t - d.task_begin - 1)
        return fail(SKYOPT_EINVAL, "dag %d: chain parent must be the previous task", i);
    }
  }
  if (pb->n_reservations < 0 || (pb->n_reservations > 0 && !pb->reservations))
    return fail(SKYOPT_EINVAL, "bad reservation table");
  for (int i = 0; i < pb->n_reservations; ++i) {
    const SkyoptReservation &r = pb->reservations[i];
    if (r.cloud < 0 || r.cloud >= C) return fail(SKYOPT_EINVAL, "reservation %d: bad cloud %d", i, r.cloud);
    if (r.inst_id < cat->cloud_inst_offsets[r.cloud] || r.inst_id >= cat->cloud_inst_offsets[r.cloud + 1])
      return fail(SKYOPT_EINVAL, "reservation %d: instance id %d is not of cloud %d", i, r.inst_id, r.cloud);
    if (r.zone_id < 0 || r.zone_id >= cat->cloud_n_zones[r.cloud])
      return fail(SKYOPT_EINVAL, "reservation %d: bad zone id %d", i, r.zone_id);
    if (r.available <= 0) return fail(SKYOPT_EINVAL, "reservation %d: available must be > 0", i);
    if (i > 0) {
      const SkyoptReservation &q = pb->reservations[i - 1];
      const bool ordered = q.cloud < r.cloud || (q.cloud == r.cloud && (q.inst_id < r.inst_id ||
                           (q.inst_id == r.inst_id && q.zone_id < r.zone_id)));
      if (!ordered) return fail(SKYOPT_EINVAL, "reservation %d: table not sorted by (cloud, inst_id, zone_id) or not unique", i);
    }
  }
  return 0;
}

// Sizes, scan grouping and offsets; fills the host staging copy.
int build_plan(SkyoptCatalog *cat, const SkyoptProblem *pb, Ctx *x, Plan &P) {
  const int C = cat->dev.n_clouds;
  P.nq = pb->n_queries; P.nsets = pb->n_acc_sets; P.ns = pb->n_slots;
  P.nt = pb->n_tasks; P.np = pb->n_parents; P.ntar = pb->n_tariffs;
  P.nb = pb->n_blocked; P.nd = pb->n_dags; P.nres = pb->n_reservations;

  std::vector<std::vector<int>> by_cloud(C);
  for (int i = 0; i < P.nq; ++i) by_cloud[pb->queries[i].cloud].push_back(i);
  // Scan units: a (cloud, tile class) pair with its own query groups. Up to 32
  // queries share one pass over a unit's rows. A row chunk that many queries
  // match at once is scored query by query by one warp, so groups are cut
  // early when the expected number of queries surviving the zone-map test per
  // chunk (the class's flag density; accelerator and fixed-host queries are
  // selective by key) reaches kDenseCut: the dense tiles of the catalog are
  // then spread over more blocks instead of forming the tail of the launch,
  // while the sparse tiles keep all queries fused.
  // Round-2 fast path: plain argmin queries (no list / fuzzy tables), class
  // dictionaries that fit shared memory, single-key accelerator slots.
  P.fast = false;
  if (cat->fast_ok && (cat->scan_mode == 0 || cat->scan_mode == 6)) {
    bool ok = true;
    for (int i = 0; i < P.nq && ok; ++i)
      if (pb->queries[i].qflags & (SKYOPT_Q_LIST | SKYOPT_Q_FUZZY)) ok = false;
    for (int s = 0; s < P.ns && ok; ++s) {
      const int set = pb->slots[s].acc_set;
      if (set < 0) continue;
      int bits = 0;
      const uint32_t *w = pb->acc_sets + (size_t)set * SKYOPT_ACC_SET_WORDS;
      for (int k = 0; k < SKYOPT_ACC_SET_WORDS; ++k) bits += __builtin_popcount(w[k]);
      if (bits > 1) ok = false;  // several spellings of one accelerator: merge needs a sort
    }
    for (int t = 0; t < P.nt && ok; ++t)
      if (pb->tasks[t].slot_end - pb->tasks[t].slot_begin > kFastMaxTaskSlots) ok = false;
    P.fast = ok;
  }
  static const float kDenseCut = [] {
    const char *e = getenv("SKYOPT_DENSE_CUT");
    return e ? (float)atof(e) : 3.0f;
  }();
  // n_tiles: tiles of the unit; n_blocks: blocks of each of its groups; tpb:
  // tiles per block (strided over the unit's tile list)
  struct Unit { int cloud, klass, n_tiles, n_blocks, tpb, list0, tile0; std::vector<int> cuts; };
  auto make_units = [&](int rpt, int tpb, bool by_class, std::vector<Unit> &units,
                        float target_pairs = 0.f) {
    long long blocks = 0;
    units.clear();
    const int tile = kScanThreads * rpt;
    const int r = rpt == 4 ? 2 : (rpt == 2 ? 1 : 0);
    for (int c = 0; c < C; ++c) {
      const auto &qs = by_cloud[c];
      if (qs.empty()) continue;
      const int rows = cat->cloud_row_offsets[c + 1] - cat->cloud_row_offsets[c];
      for (int k = 0; k < (by_class ? 2 : 1); ++k) {
        Unit u; u.cloud = c; u.klass = k; u.tpb = tpb;
        const float *density;
        if (by_class) {
          const SkyoptCatalog::TileClass &tc = cat->tile_class[r][c][k];
          if (tc.n_tiles == 0) continue;
          u.n_tiles = tc.n_tiles; u.list0 = tc.list0; u.tile0 = tc.tile0; density = tc.density.data();
        } else {
          u.n_tiles = (rows + tile - 1) / tile; u.list0 = -1; u.tile0 = 0;
          density = cat->flag_density[c].data();
        }
        u.cuts.push_back(0);
        float dens = 0.f, dmax = 0.f; int n = 0;
        for (size_t i = 0; i < qs.size(); ++i) {
          const SkyoptQuery &q = pb->queries[qs[i]];
          float dq = density[(q.flags_require | SKYOPT_F_VALID) & 0xFFu];
          if ((q.qflags & SKYOPT_Q_ACC) || q.group != 0) dq *= 0.05f;
          if (n > 0 && (n == kQChunk || dens + dq > kDenseCut)) {
            u.cuts.push_back((int)i); dens = 0.f; n = 0;
          }
          dens += dq; ++n;
          dmax = std::max(dmax, dens);
        }
        u.cuts.push_back((int)qs.size());
        if (target_pairs > 0.f) {
          // queue form: as many tiles per block (at most 32: one tested chunk
          // per thread) as keep the expected number of surviving (chunk,
          // query) pairs of the unit's densest group near the target
          const float per_tile = (float)(tile / 128) * std::max(dmax, 1e-3f);
          u.tpb = std::min(32, std::max(1, (int)(target_pairs / per_tile)));
        }
        u.n_blocks = (u.n_tiles + u.tpb - 1) / u.tpb;
        blocks += (long long)u.n_blocks * (long long)(u.cuts.size() - 1);
        units.push_back(std::move(u));
      }
    }
    return blocks;
  };
  // One tile of 256*RPT rows per block (rows go straight to registers), with
  // smaller tiles when there is too little work to cover all SMs. The TMA
  // streaming kernel (several 1024-row tiles per block through shared memory)
  // is selectable (SKYOPT_SCAN_MODE=stream / skyopt_catalog_set_scan_mode):
  // on B200 it is slower for this workload -- scoring, not the row stream,
  // is the critical path and fewer, longer-lived blocks overlap it worse
  // (profiles/round1_scan_experiments.md) -- so "auto" never picks it.
  P.rpt = 4; P.tpb = 1; P.stream = false;
  std::vector<Unit> units;
  const long long wave = 2ll * cat->sm_count;
  // fast path: groups of <= 32 queries per (cloud, price column), cut into
  // pieces of consecutive 128-row chunks for a persistent grid
  std::vector<Scan2Group> groups2;
  std::vector<int> order2;  // scan order -> caller's query index
  std::vector<char> gate_used(std::max(P.nq, 1), 0);
  for (int sl = 0; sl < P.ns; ++sl) if (pb->slots[sl].gate_query >= 0) gate_used[pb->slots[sl].gate_query] = 1;
  if (P.fast) {
    long long visits = 0;
    for (int c = 0; c < C; ++c)
      for (int col = 0; col < 2; ++col) {
        std::vector<int> qs;
        for (int qi : by_cloud[c]) if ((pb->queries[qi].price_col ? 1 : 0) == col) qs.push_back(qi);
        for (size_t b = 0; b < qs.size(); b += kQChunk) {
          Scan2Group G{};
          G.cloud = c; G.col = col; G.q_begin = (int)order2.size();
          G.q_count = (int)std::min<size_t>(kQChunk, qs.size() - b);
          G.n_cm = cat->n_cm[c]; G.n_fa = cat->n_fa[c]; G.n_rz = cat->n_rz[c];
          G.cm_off = cat->cm_off[c]; G.fa_off = cat->fa_off[c]; G.rz_off = cat->rz_off[c];
          G.chunk0 = cat->cloud_row_offsets[c] / kZoneRows;
          G.n_chunks = cat->cloud_row_offsets[c + 1] / kZoneRows - G.chunk0;
          for (int k = 0; k < G.q_count; ++k) { order2.push_back(qs[b + k]); if (gate_used[qs[b + k]]) G.need_any = 1; }
          if (P.ns == 0) G.need_any = 1;  // skyopt_scan: every result carries any_stage1
          if (G.n_chunks > 0) groups2.push_back(G);
          visits += G.n_chunks;
          P.cap_fa = std::max(P.cap_fa, (uint32_t)G.n_fa); P.cap_cm = std::max(P.cap_cm, (uint32_t)G.n_cm);
          P.cap_rz = std::max(P.cap_rz, (uint32_t)G.n_rz);
        }
      }
    P.cap_fa = (P.cap_fa + 3u) & ~3u; P.cap_cm = (P.cap_cm + 3u) & ~3u; P.cap_rz = (P.cap_rz + 3u) & ~3u;
    P.scan2_smem = scan2_smem_bytes(P.cap_fa, P.cap_cm, P.cap_rz);
    P.step_smem = std::max(P.scan2_smem, std::max(sizeof(PlaceSmem), sizeof(ChainSmem))) + 16;
    int per_sm = kScanBlocksPerSM;
    {
      static std::mutex occ_mu;
      std::lock_guard<std::mutex> g(occ_mu);
      // the separate-launch scan (4 blocks of 61 registers per SM) has more
      // resident blocks than the fused kernel (3)
      const cudaError_t oe = cat->split
          ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, scan2_kernel, kScanThreads, P.scan2_smem)
          : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, step_kernel, kScanThreads, P.step_smem);
      if (oe != cudaSuccess || per_sm < 1) per_sm = 1;
    }
    static const int grid_cap = [] { const char *e = getenv("SKYOPT_SCAN2_BLOCKS_PER_SM"); return e ? atoi(e) : 0; }();
    if (grid_cap > 0) per_sm = std::min(per_sm, grid_cap);
    const long long resident = (long long)per_sm * cat->sm_count;
    // Pieces of consecutive chunks: at most one per resident block (a second
    // piece of another group would re-stage and rebuild the tables), at least
    // `min_piece` chunks each.
    static const int min_piece = [] { const char *e = getenv("SKYOPT_SCAN2_MIN_PIECE"); return e ? std::max(1, atoi(e)) : 8; }();
    const long long spare = std::max<long long>(0, resident - (long long)groups2.size());
    int piece0 = 0;
    for (Scan2Group &G : groups2) {
      long long k = 1 + (visits > 0 ? spare * G.n_chunks / visits : 0);
      k = std::min<long long>(k, std::max<long long>(1, G.n_chunks / min_piece));
      G.piece0 = piece0; G.index = (int)(&G - groups2.data());
      G.n_pieces = (int)std::max<long long>(1, std::min<long long>(k, G.n_chunks));
      piece0 += G.n_pieces;
      P.layout_rows += (long long)G.n_chunks * kZoneRows;
    }
    P.step_grid = (int)std::min<long long>(resident, std::max<long long>(piece0, P.nt));
    P.n_groups2 = (int)groups2.size(); P.n_pieces = piece0;
    P.scan2_grid = (int)std::min<long long>(resident, std::max(P.n_pieces, 1));
    P.chain_dags = true;
    for (int d = 0; d < P.nd; ++d)
      if (!pb->dags[d].is_chain || pb->dags[d].task_end - pb->dags[d].task_begin > kFastTasks) P.chain_dags = false;
    P.n_groups = 0; P.nsq = (int)order2.size();
  } else
  if (cat->scan_mode == 2 || cat->scan_mode == 3) {
    P.stream = true;
    const long long tiles4 = make_units(4, 1, false, units);
    P.tpb = (int)std::max<long long>(1, (tiles4 + wave - 1) / wave);
    if (cat->scan_mode == 3) P.tpb = 3;  // tests: force the multi-tile loop
    if (const char *t = getenv("SKYOPT_TPB")) P.tpb = std::max(1, atoi(t));
    make_units(4, P.tpb, false, units);
  } else {
    static const float queue_target = [] { const char *e = getenv("SKYOPT_SCAN_Q"); return e ? (float)atof(e) : -1.f; }();
    if (const char *r = getenv("SKYOPT_RPT")) {
      const int v = atoi(r);
      if (v == 1 || v == 2 || v == 4) P.rpt = v;
      make_units(P.rpt, 1, true, units);
    } else if (cat->scan_mode < 4 &&
               (cat->scan_mode == 1 || queue_target == 0.f || make_units(4, 1, true, units) < 3 * wave)) {
      // few tiles: one per block, smaller ones when they do not cover the SMs
      if (make_units(4, 1, true, units) < wave) {
        P.rpt = 2;
        if (make_units(2, 1, true, units) < wave) { P.rpt = 1; make_units(1, 1, true, units); }
      }
    } else {
      // Queue form (scan_queue_kernel): blocks own several tiles and their
      // warps share the surviving (chunk, query) pairs. The target number of
      // pairs per block is the smallest that lets the whole grid be resident
      // at once (kScanBlocksPerSM blocks per SM, a tenth left free): a second
      // wave would start behind blocks that live 8-12 us
      // (profiles/round1_scan_experiments.md).
      P.queue = true;
      const long long resident = (long long)(0.9 * kScanBlocksPerSM * cat->sm_count);
      float target = queue_target > 0.f ? queue_target : 16.f;
      if (cat->scan_mode == 5) target = 1e9f;  // tests: 32 tiles per block everywhere
      while (make_units(4, 1, true, units, target) > resident && queue_target <= 0.f && target < 256.f)
        target = target < 64.f ? target + 8.f : target * 1.5f;
    }
    // dense units first (their blocks live longest) when asked; with the
    // permuted launch order it makes no measurable difference
    static const bool dense_first = [] { const char *e = getenv("SKYOPT_DENSE_FIRST"); return e && atoi(e) != 0; }();
    if (dense_first)
      std::stable_sort(units.begin(), units.end(), [](const Unit &a, const Unit &b) { return a.klass > b.klass; });
  }
  const int tile = kScanThreads * P.rpt;
  if (!P.fast) { P.n_groups = 0; P.nsq = 0; }
  std::vector<int> cloud_tiles(C, 0);  // partial slots of one query of the cloud
  for (const Unit &u : units) {
    P.n_groups += (int)u.cuts.size() - 1;
    P.nsq += (int)by_cloud[u.cloud].size();
    cloud_tiles[u.cloud] += u.n_blocks;
  }

  // candidate capacity: every slot can at most expand to its cloud's largest
  // instance-type / accelerator group
  std::vector<int64_t> slot_off(P.ns);
  int64_t cap = 0;
  for (int s = 0; s < P.ns; ++s) { slot_off[s] = cap; cap += cat->cloud_group_cap[pb->slots[s].cloud]; }
  P.cand_cap = cap;

  // partial / table offsets
  std::vector<int32_t> pbase(P.nq), pcount(P.nq);
  std::vector<int64_t> lbase(P.nq, 0), fbase(P.nq, 0);
  int64_t npart = 0, nlist = 0, nfuzzy = 0;
  P.scan_rows = 0;
  for (int i = 0; i < P.nq; ++i) {
    const SkyoptQuery &q = pb->queries[i];
    const int rows = cat->cloud_row_offsets[q.cloud + 1] - cat->cloud_row_offsets[q.cloud];
    pcount[i] = cloud_tiles[q.cloud];
    if (npart + pcount[i] > 0x7FFFFFFFll) return fail(SKYOPT_ELIMIT, "too many scan partials");
    pbase[i] = (int32_t)npart; npart += pcount[i];
    P.scan_rows += rows;
    if (q.qflags & SKYOPT_Q_LIST) { lbase[i] = nlist; nlist += cat->cloud_inst_offsets[q.cloud + 1] - cat->cloud_inst_offsets[q.cloud]; }
    if (q.qflags & SKYOPT_Q_FUZZY) { fbase[i] = nfuzzy; nfuzzy += cat->dev.n_acc_keys; }
  }
  P.n_partials = npart; P.list_entries = nlist; P.fuzzy_entries = nfuzzy;

  Carver sizing(nullptr);
  carve_inputs(P, sizing);
  P.in_bytes = align_up(sizing.off);
  carve_rest(P, sizing);
  P.total_bytes = align_up(sizing.off);
  int rc = ensure(x, P.total_bytes, std::max(P.in_bytes, P.out_bytes));
  if (rc) return rc;

  // host staging copy of the input region
  Carver h(x->hbuf);
  carve_inputs(P, h);
  memcpy(P.queries, pb->queries, sizeof(SkyoptQuery) * P.nq);
  if (P.nsets) memcpy(P.acc_sets, pb->acc_sets, sizeof(uint32_t) * SKYOPT_ACC_SET_WORDS * P.nsets);
  if (P.ns) memcpy(P.slots, pb->slots, sizeof(SkyoptSlot) * P.ns);
  if (P.nt) memcpy(P.tasks, pb->tasks, sizeof(SkyoptTask) * P.nt);
  if (P.np) memcpy(P.parents, pb->parents, sizeof(int32_t) * P.np);
  if (P.ntar) memcpy(P.tariffs, pb->tariffs, sizeof(double) * P.ntar);
  if (P.nb) memcpy(P.blocked, pb->blocked, sizeof(SkyoptBlocked) * P.nb);
  if (P.nd) memcpy(P.dags, pb->dags, sizeof(SkyoptDag) * P.nd);
  if (P.nres) memcpy(P.res, pb->reservations, sizeof(SkyoptReservation) * P.nres);
  memcpy(P.partial_base, pbase.data(), sizeof(int32_t) * P.nq);
  memcpy(P.partial_count, pcount.data(), sizeof(int32_t) * P.nq);
  memcpy(P.list_base, lbase.data(), sizeof(int64_t) * P.nq);
  memcpy(P.fuzzy_base, fbase.data(), sizeof(int64_t) * P.nq);
  if (P.ns) memcpy(P.slot_off, slot_off.data(), sizeof(int64_t) * P.ns);
  // task candidate capacity = sum of its slots' capacities
  {
    int64_t off = 0;
    for (int t = 0; t < P.nt; ++t) {
      P.task_off[t] = off;
      for (int s = pb->tasks[t].slot_begin; s < pb->tasks[t].slot_end; ++s)
        off += cat->cloud_group_cap[pb->slots[s].cloud];
    }
    P.task_off[P.nt] = off;
    if (off > P.cand_cap) {
      // slots shared by several tasks would overflow the task arrays
      return fail(SKYOPT_EINVAL, "a slot belongs to more than one task");
    }
  }
  for (int t = 0; t < P.nt; ++t) P.task_dag[t] = 0;
  for (int d = 0; d < P.nd; ++d)
    for (int t = pb->dags[d].task_begin; t < pb->dags[d].task_end; ++t) P.task_dag[t] = d;
  auto fill_record = [&](ScanQuery &R, int qi) {
    const SkyoptQuery &q = pb->queries[qi];
    memset(&R, 0, sizeof(R));
    R.s = make_query_s(q);
    R.qid = qi;
    R.list_base = lbase[qi];
    R.fuzzy_base = fbase[qi];
    uint32_t lo32 = 0, hi32 = 0;
    const int set_idx[2] = {(q.qflags & SKYOPT_Q_ACC) ? q.acc_set : -1,
                            (q.qflags & SKYOPT_Q_FUZZY) ? q.fuzzy_set : -1};
    for (int which = 0; which < 2; ++which) {
      if (set_idx[which] < 0) continue;
      const uint32_t *src = pb->acc_sets + (size_t)set_idx[which] * SKYOPT_ACC_SET_WORDS;
      for (int w = 0; w < SKYOPT_ACC_SET_WORDS; ++w) {
        R.set[which][w] = src[w];
        if (w & 1) hi32 |= src[w]; else lo32 |= src[w];
      }
    }
    // 64-bit signature (key id mod 64) of the keys the query can match
    R.s.sig_lo = (q.qflags & SKYOPT_Q_ACC) ? lo32 : 0xFFFFFFFFu;
    R.s.sig_hi = (q.qflags & SKYOPT_Q_ACC) ? hi32 : 0xFFFFFFFFu;
  };
  if (P.fast) {
    for (int i = 0; i < P.nsq; ++i) fill_record(P.squeries[i], order2[i]);
    memcpy(P.groups2, groups2.data(), sizeof(Scan2Group) * groups2.size());
    memset(P.best_rank, 0xFF, sizeof(uint32_t) * 2 * P.nq);
    memset(P.any_in, 0, sizeof(uint32_t) * 2 * P.nq);
    if (P.nd) memset(P.dag_done, 0, sizeof(int32_t) * P.nd);
    if (P.n_groups2) memset(P.group_ready, 0, sizeof(unsigned int) * 2 * P.n_groups2);
    // what a task block / a slot needs, in one record each
    for (int t = 0; t < P.nt; ++t) {
      const SkyoptDag &D = pb->dags[P.task_dag[t]];
      PlaceTask &T = P.ptasks[t];
      T.slot_begin = pb->tasks[t].slot_begin; T.slot_end = pb->tasks[t].slot_end;
      T.blocked_begin = D.blocked_begin; T.blocked_end = D.blocked_end;
      T.minimize_cost = D.minimize_cost; T.pad_[0] = T.pad_[1] = T.pad_[2] = 0;
    }
    for (int sl = 0; sl < P.ns; ++sl) {
      const SkyoptSlot &S = pb->slots[sl];
      SlotAux &X = P.saux[sl];
      memset(&X, 0, sizeof(X));
      X.max_price = 1.0 / 0.0;
      if (S.query >= 0) {
        const SkyoptQuery &Q = pb->queries[S.query];
        X.rec_base = cat->cloud_row_offsets[Q.cloud]; X.qcol = Q.price_col ? 1 : 0; X.max_price = Q.max_price;
      }
      X.cloud_r0 = cat->cloud_row_offsets[S.cloud]; X.cloud_r1 = cat->cloud_row_offsets[S.cloud + 1];
      X.has_zones = cat->cloud_n_zones[S.cloud] > 0 ? 1 : 0;
      X.acc_list_key = -1;
      if (S.acc_set >= 0) {
        const uint32_t *w = pb->acc_sets + (size_t)S.acc_set * SKYOPT_ACC_SET_WORDS;
        for (int k = 0; k < SKYOPT_ACC_SET_WORDS && X.acc_list_key < 0; ++k)
          if (w[k]) X.acc_list_key = (int16_t)(32 * k + __builtin_ctz(w[k]));
      }
    }
  }
  int g = 0, qpos = 0, block0 = 0;
  P.pass_rows = 0;
  std::vector<int> unit_pbase(C, 0);  // partial slots used by earlier units of the cloud
  for (int c = 0; c < C; ++c) {
    // algorithmic passes: the minimum (32 fused queries per pass over the
    // cloud's rows), whatever grouping is chosen
    const int rows = cat->cloud_row_offsets[c + 1] - cat->cloud_row_offsets[c];
    P.pass_rows += (int64_t)rows * (int64_t)((by_cloud[c].size() + kQChunk - 1) / kQChunk);
  }
  for (const Unit &u : units) {
    const int c = u.cloud;
    const auto &qs = by_cloud[c];
    const int rows = cat->cloud_row_offsets[c + 1] - cat->cloud_row_offsets[c];
    const int total_tiles = (rows + tile - 1) / tile;
    const int tiles = u.n_blocks;  // blocks of each group of the unit
    for (size_t ci = 0; ci + 1 < u.cuts.size(); ++ci) {
      const size_t b = (size_t)u.cuts[ci];
      const int n = u.cuts[ci + 1] - u.cuts[ci];
      ScanGroup G{};
      G.row_begin = cat->cloud_row_offsets[c];
      G.row_end = cat->cloud_row_offsets[c + 1];
      G.q_begin = qpos; G.q_count = n; G.block0 = block0; G.n_tiles = tiles;
      G.tiles_per_block = u.tpb; G.total_tiles = P.stream ? total_tiles : u.n_tiles;
      G.list0 = u.list0; G.tile0 = u.tile0;
      for (int k = 0; k < n; ++k) {
        const int qi = qs[b + k];
        const SkyoptQuery &q = pb->queries[qi];
        G.need |= q.price_col ? 2u : 1u;
        if (q.qflags & SKYOPT_Q_FUZZY) G.need |= 1u;
        // the staged record: constraint vector, offsets and key bitmasks
        ScanQuery &R = P.squeries[qpos + k];
        fill_record(R, qi);
        R.partial_base = pbase[qi] + unit_pbase[c];
        QueryTest &T = P.qtests[qpos + k];
        T.req_flags = R.s.req_flags; T.grp_bit = R.s.grp_bit;
        T.sig_lo = R.s.sig_lo; T.sig_hi = R.s.sig_hi;
        T.qflags = R.s.qflags; T.price_col = (uint32_t)(R.s.price_col ? 1 : 0);
        T.partial_base = R.partial_base; T.pad_ = 0;
      }
      P.groups[g++] = G;
      qpos += n; block0 += tiles;
    }
    unit_pbase[c] += tiles;
  }
  P.n_blocks = block0;

  const ScanGroup *host_groups = P.groups;
  P.host_groups2 = P.groups2;
  // device views
  Carver d(x->dbuf);
  carve_inputs(P, d);
  carve_rest(P, d);
  P.host_groups = host_groups;  // pinned staging copy stays valid for the call
  return 0;
}

struct Timeline { float scan_ms = 0, expand_ms = 0, solve_ms = 0; };

// Round-2 path: scan2 -> [finalize2] -> place -> solve. `first` = the result
// arrays were just initialised by the H2D copy of the input region; later
// iterations of the device-resident timing loop reset them with one memset.
int enqueue_fast(SkyoptCatalog *cat, Ctx *x, const Plan &P, bool solve, bool want_scan_results) {
  cudaStream_t st = x->stream;
  CU(cudaEventRecord(x->ev[1], st));
  Scan2Args sa{};
  sa.cat = cat->dev; sa.f = cat->fast; sa.squeries = P.squeries; sa.groups = P.groups2;
  sa.n_groups = P.n_groups2; sa.n_pieces = P.n_pieces;
  // fused launches alternate between the two copies of the scan results
  const size_t par = (size_t)(P.parity & 1), oth = par ^ 1;
  uint32_t *best_rank = P.best_rank + par * P.nq, *any_in = P.any_in + par * P.nq;
  sa.best_rank = best_rank; sa.any1 = any_in;
  sa.zero_flag = P.err_out; sa.cap_fa = P.cap_fa; sa.cap_cm = P.cap_cm; sa.cap_rz = P.cap_rz;
  sa.trace = x->trace; sa.shared_tables = nullptr; sa.group_ready = nullptr;
  for (int i = 0; i < std::min(P.n_groups2, kInlineGroups2); ++i) {
    sa.inline_groups[i] = P.host_groups2[i]; sa.inline_piece0[i] = P.host_groups2[i].piece0;
  }
  static const bool noprune_env = [] { const char *e = getenv("SKYOPT_NOPRUNE"); return e && atoi(e) != 0; }();
  sa.noprune = (noprune_env || cat->noprune) ? 1u : 0u;
  sa.force_any = (want_scan_results || !solve) ? 1u : 0u;
  ExpandOut ex0{P.slot_count, P.slot_inst, P.cand_region, P.cand_zone, P.cand_pa, P.cand_pb};
  SolveIn in0{P.slots, P.tasks, P.parents, P.tariffs, P.blocked, P.dags, P.slot_off, P.task_off, ex0, 0, P.res, P.nres};
  SolveWork w0{P.tc_ref, P.tc_slot, P.tc_cloud, P.tc_hourly, P.tc_value, P.dp, P.back};
  static const bool split_env = [] { const char *e = getenv("SKYOPT_SPLIT"); return e && atoi(e) != 0; }();
  P.ran_fused = false;
  if (solve && !want_scan_results && P.nt && cat->coop && !cat->split && !split_env) {
    // ---- the whole step in one cooperative launch
    StepArgs sp{};
    sp.scan = sa;
    static const int exp_flags = [] { const char *e = getenv("SKYOPT_EXP"); return e ? atoi(e) : 0; }();
    if (!(exp_flags & 2)) { sp.scan.shared_tables = P.shared_tables; sp.scan.group_ready = P.group_ready + par * P.n_groups2; }
    sp.next_best_rank = P.best_rank + oth * P.nq; sp.next_any1 = P.any_in + oth * P.nq;
    sp.next_group_ready = P.group_ready + oth * P.n_groups2;
    if (exp_flags & 4) sp.scan.noprune |= 4u;  // experiment: spin without nanosleep
    sp.force_full = ((exp_flags & 8) ? 1 : 0) | ((exp_flags & 16) ? 2 : 0);   // test knob: evaluate every candidate in the chain DP
    sp.place.cat = cat->dev; sp.place.f = cat->fast; sp.place.ptasks = P.ptasks; sp.place.saux = P.saux;
    sp.place.best_rank = best_rank; sp.place.any1 = any_in; sp.place.acc_sets = P.acc_sets;
    sp.place.in = in0; sp.place.w = w0; sp.place.task_n = P.task_n; sp.place.trace = x->trace;
    sp.place.task_mv = P.task_mv;
    sp.out = SolveOut{P.chosen, P.chosen_index, P.task_n, P.dagres, x->trace};
    sp.task_dag = P.task_dag; sp.n_tasks = P.nt; sp.do_solve = P.chain_dags ? 1 : 0;
    sp.dag_done = P.dag_done; sp.sync = x->sync;
    if (x->sync_total > 0x70000000u - (unsigned)P.step_grid) {
      CU(cudaMemsetAsync(x->sync, 0, sizeof(unsigned int), st));
      x->sync_total = 0;
    }
    sp.sync_target = x->sync_total + (unsigned)P.step_grid;
    sp.n_queries = P.nq;
    sp.in_base = x->dbuf; sp.in_lines = (int64_t)((P.in_bytes + 127) / 128);
    void *args[] = {&sp};
    // step_kernel leaves best_rank / any_in reset for the next launch: no
    // memset, no event between ev[1] and ev[4] (each costs microseconds here)
    cudaError_t le = cudaLaunchCooperativeKernel((const void *)step_kernel, dim3(P.step_grid), dim3(kScanThreads),
                                                 args, P.step_smem, st);
    if (le == cudaSuccess) {
      x->sync_total += (unsigned)P.step_grid;
      P.parity ^= 1;
      if (!P.chain_dags && P.nd) {
        SolveOut out{P.chosen, P.chosen_index, P.task_n, P.dagres, x->trace};
        solve_kernel<<<P.nd, kSolveThreads, 0, st>>>(cat->dev, in0, w0, out);
        CU(cudaGetLastError());
      }
      CU(cudaEventRecord(x->ev[4], st));
      P.ran_fused = true;
      return 0;
    }
    (void)cudaGetLastError();  // not launched (too large for this device): separate launches below
  }
  if (P.nq) {
    if (!P.fresh_inputs) {
      CU(cudaMemsetAsync(best_rank, 0xFF, sizeof(uint32_t) * P.nq, st));
      CU(cudaMemsetAsync(any_in, 0, sizeof(uint32_t) * P.nq, st));
    }
    CU(cudaEventRecord(x->ev[6], st));
    if (P.n_pieces) {
      scan2_kernel<<<P.scan2_grid, kScanThreads, P.scan2_smem, st>>>(sa);
      CU(cudaGetLastError());
    }
    CU(cudaEventRecord(x->ev[7], st));
    if (want_scan_results || !solve) {
      finalize2_kernel<<<(P.nq + 127) / 128, 128, 0, st>>>(cat->dev, cat->fast, P.nq, P.queries,
                                                          best_rank, any_in, P.finals, P.any1);
      CU(cudaGetLastError());
    }
  }
  CU(cudaEventRecord(x->ev[2], st));
  if (!solve) return 0;
  if (!P.n_pieces) CU(cudaMemsetAsync(P.err_out, 0, sizeof(int32_t), st));
  ExpandOut ex{P.slot_count, P.slot_inst, P.cand_region, P.cand_zone, P.cand_pa, P.cand_pb};
  SolveIn in{P.slots, P.tasks, P.parents, P.tariffs, P.blocked, P.dags, P.slot_off, P.task_off, ex, 0, P.res, P.nres};
  SolveWork w{P.tc_ref, P.tc_slot, P.tc_cloud, P.tc_hourly, P.tc_value, P.dp, P.back};
  if (P.nt) {
    PlaceArgs pa{};
    pa.cat = cat->dev; pa.f = cat->fast; pa.ptasks = P.ptasks; pa.saux = P.saux; pa.best_rank = best_rank;
    pa.any1 = any_in; pa.acc_sets = P.acc_sets; pa.in = in; pa.w = w;
    pa.task_n = P.task_n; pa.trace = x->trace; pa.task_mv = nullptr;
    place_kernel<<<P.nt, kScanThreads, sizeof(PlaceSmem), st>>>(pa);
    CU(cudaGetLastError());
  }
  CU(cudaEventRecord(x->ev[3], st));
  if (P.nd) {
    SolveOut out{P.chosen, P.chosen_index, P.task_n, P.dagres, x->trace};
    solve_kernel<<<P.nd, kSolveThreads, 0, st>>>(cat->dev, in, w, out);
    CU(cudaGetLastError());
  }
  CU(cudaEventRecord(x->ev[4], st));
  return 0;
}

// Enqueue K1..K3 on the context's stream. Events ev[1..4] bracket the phases.
int enqueue_kernels(SkyoptCatalog *cat, Ctx *x, const Plan &P, bool solve,
                    bool want_scan_results = true) {
  cudaStream_t st = x->stream;
  if (P.fast) return enqueue_fast(cat, x, P, solve, want_scan_results);
  CU(cudaEventRecord(x->ev[1], st));
  if (P.nq) {
    CU(cudaMemsetAsync(P.gbest, 0xFF, sizeof(unsigned long long) * P.nsq, st));
    if (P.list_entries) CU(cudaMemsetAsync(P.list_min, 0xFF, sizeof(unsigned long long) * P.list_entries, st));
    if (P.fuzzy_entries) CU(cudaMemsetAsync(P.fuzzy_min, 0xFF, sizeof(unsigned long long) * P.fuzzy_entries, st));
    if (P.n_blocks) {
      ScanArgs sa{};
      sa.cat = cat->dev; sa.squeries = P.squeries; sa.qtests = P.qtests; sa.groups = P.groups;
      sa.n_groups = P.n_groups; sa.partials = P.partials;
      sa.list_min = P.list_min; sa.fuzzy_min = P.fuzzy_min; sa.gbest = P.gbest;
      sa.zero_flag = P.err_out; sa.tile_list = cat->d_tile_list;
      for (int i = 0; i < std::min(P.n_groups, kInlineGroups); ++i) { sa.inline_groups[i] = P.host_groups[i]; sa.inline_block0[i] = P.host_groups[i].block0; }
      sa.n_blocks = P.n_blocks;
      sa.debug = 0;
      if (const char *dbg = getenv("SKYOPT_DEBUG")) sa.debug = (uint32_t)atoi(dbg);
      sa.qsplit = 2;
      if (const char *qs = getenv("SKYOPT_QSPLIT")) sa.qsplit = (uint32_t)std::max(1, atoi(qs));
      static unsigned long long *tl = nullptr; static int tl_blocks = 0;
      if (sa.debug & 2u) {
        if (tl_blocks < P.n_blocks) { if (tl) cudaFree(tl); CU(cudaMalloc(&tl, (size_t)P.n_blocks * 64 + 1024)); tl_blocks = P.n_blocks; }
        sa.timeline = tl;
        CU(cudaMemsetAsync(tl + (size_t)P.n_blocks * 8, 0, 1024, st));
        if (const char *e = getenv("SKYOPT_TRACE_VB")) sa.trace_vb = (uint32_t)atoi(e);
        if (const char *e = getenv("SKYOPT_TRACE_WARP")) sa.trace_warp = (uint32_t)atoi(e);
      }
      sa.perm_mul = 1;
      static const bool permute = [] { const char *e = getenv("SKYOPT_PERM"); return !e || atoi(e) != 0; }();
      if (permute) for (uint32_t cand : {7919u, 104729u, 1299709u, 15485863u}) {
        uint64_t x = cand, y = (uint64_t)P.n_blocks;  // gcd
        while (y) { const uint64_t t = x % y; x = y; y = t; }
        if (x == 1) { sa.perm_mul = cand; break; }
      }
      CU(cudaEventRecord(x->ev[6], st));
      if (P.stream)
        scan_stream_kernel<<<P.n_blocks, kScanThreads, kStreamStages * sizeof(StreamStage), st>>>(sa);
      else if (P.queue) scan_queue_kernel<<<P.n_blocks, kScanThreads, 0, st>>>(sa);
      else if (P.rpt == 4) scan_kernel<4><<<P.n_blocks, kScanThreads, 0, st>>>(sa);
      else if (P.rpt == 2) scan_kernel<2><<<P.n_blocks, kScanThreads, 0, st>>>(sa);
      else scan_kernel<1><<<P.n_blocks, kScanThreads, 0, st>>>(sa);
      CU(cudaGetLastError());
      CU(cudaEventRecord(x->ev[7], st));
      if (sa.debug & 2u) {
        // profiling experiment: dump the per-block timeline of this launch
        std::vector<unsigned long long> h((size_t)P.n_blocks * 8 + 128);
        CU(cudaStreamSynchronize(st));
        CU(cudaMemcpy(h.data(), sa.timeline, h.size() * 8, cudaMemcpyDeviceToHost));
        if (const char *path = getenv("SKYOPT_TIMELINE")) {
          if (FILE *f = fopen(path, "wb")) { fwrite(h.data(), 8, h.size(), f); fclose(f); }
        }
      }
    }
    if (want_scan_results || !solve) {
      const int fblocks = (P.nq * 32 + 255) / 256;
      finalize_kernel<<<fblocks, 256, 0, st>>>(cat->dev, P.nq, P.partial_base,
                                               P.partial_count, P.partials, P.finals,
                                               P.any1, P.err_out);
      CU(cudaGetLastError());
    }
  }
  CU(cudaEventRecord(x->ev[2], st));
  if (!solve) return 0;
  if (!P.n_blocks) CU(cudaMemsetAsync(P.err_out, 0, sizeof(int32_t), st));
  ExpandOut ex{P.slot_count, P.slot_inst, P.cand_region, P.cand_zone, P.cand_pa, P.cand_pb};
  if (P.ns) {
    const size_t smem = (size_t)cat->sort_n * 16 + (size_t)cat->max_zones * 8 +
                        (size_t)cat->max_regions * 4;
    expand_kernel<<<P.ns, 128, smem, st>>>(cat->dev, P.slots, P.partial_base,
                                           P.partial_count, P.partials,
                                           P.acc_sets, P.slot_off, cat->sort_n,
                                           cat->max_regions, cat->max_zones, ex,
                                           P.err_out);
    CU(cudaGetLastError());
  }
  CU(cudaEventRecord(x->ev[3], st));
  if (P.nd) {
    SolveIn in{P.slots, P.tasks, P.parents, P.tariffs, P.blocked, P.dags, P.slot_off, P.task_off, ex, 0, P.res, P.nres};
    SolveWork w{P.tc_ref, P.tc_slot, P.tc_cloud, P.tc_hourly, P.tc_value, P.dp, P.back};
    SolveOut out{P.chosen, P.chosen_index, P.task_n, P.dagres};
    gather_kernel<<<P.nt, kGatherThreads, 0, st>>>(cat->dev, in, w, P.task_dag, P.task_n);
    CU(cudaGetLastError());
    solve_kernel<<<P.nd, kSolveThreads, 0, st>>>(cat->dev, in, w, out);
    CU(cudaGetLastError());
  }
  CU(cudaEventRecord(x->ev[4], st));
  return 0;
}

void fill_scan_results(const SkyoptCatalog *cat, const Plan &P, const Plan &H,
                       SkyoptScanResult *results) {
  (void)cat; (void)P;
  for (int i = 0; i < H.nq; ++i) {
    SkyoptScanResult r{};
    const ScanFinal &f = H.finals[i];
    r.any_stage1 = H.any1[i] ? 1 : 0;
    r.best_row = f.row;
    r.best_inst = f.inst;
    r.best_price = f.row >= 0 ? [&] {
      uint64_t k = f.key;
      uint64_t b = (k & 0x8000000000000000ull) ? (k & 0x7FFFFFFFFFFFFFFFull) : ~k;
      double d; memcpy(&d, &b, 8); return d; }() : NAN;
    results[i] = r;
  }
}

// Host view of the output region inside the pinned buffer.
void carve_output_host(const Plan &P, char *hbuf, Plan &H) {
  H = P;
  Carver c(hbuf);
  H.finals = c.take<ScanFinal>(P.nq);
  H.any1 = c.take<uint32_t>(P.nq);
  H.slot_count = c.take<int32_t>(P.ns);
  H.slot_inst = c.take<int32_t>(P.ns);
  H.chosen = c.take<SkyoptCandidate>(P.nt);
  H.chosen_index = c.take<int32_t>(P.nt);
  H.task_n = c.take<int32_t>(P.nt);
  H.dagres = c.take<SkyoptDagResult>(P.nd);
  H.err_out = c.take<int32_t>(1);
}

int copy_solution(SkyoptCatalog *cat, Ctx *x, const Plan &P, const SkyoptProblem *pb,
                  SkyoptSolution *sol) {
  Plan H;
  carve_output_host(P, x->hbuf, H);
  if (*H.err_out)
    return fail(SKYOPT_ELIMIT, "an instance-type group exceeds the expand capacity (%d rows)", cat->sort_n);
  if (sol->scan) fill_scan_results(cat, P, H, sol->scan);
  if (sol->slot_count && P.ns) memcpy(sol->slot_count, H.slot_count, sizeof(int32_t) * P.ns);
  if (sol->slot_inst && P.ns) memcpy(sol->slot_inst, H.slot_inst, sizeof(int32_t) * P.ns);
  if (sol->chosen && P.nt) memcpy(sol->chosen, H.chosen, sizeof(SkyoptCandidate) * P.nt);
  if (sol->chosen_index && P.nt) memcpy(sol->chosen_index, H.chosen_index, sizeof(int32_t) * P.nt);
  if (sol->task_n_candidates && P.nt) memcpy(sol->task_n_candidates, H.task_n, sizeof(int32_t) * P.nt);
  if (sol->dag && P.nd) memcpy(sol->dag, H.dagres, sizeof(SkyoptDagResult) * P.nd);
  // Tasks of a failed DAG carry no plan.
  if (sol->chosen_index) {
    for (int d = 0; d < P.nd; ++d)
      if (H.dagres[d].status != 0)
        for (int t = pb->dags[d].task_begin; t < pb->dags[d].task_end; ++t) {
          sol->chosen_index[t] = -1;
          if (sol->chosen) { sol->chosen[t] = SkyoptCandidate{}; sol->chosen[t].slot = -1; sol->chosen[t].inst_id = -1; }
        }
  }
  if (sol->cand_cap > 0 && sol->candidates && sol->task_cand_offset) {
    std::vector<int64_t> off(P.nt + 1, 0);
    for (int t = 0; t < P.nt; ++t) off[t + 1] = off[t] + H.task_n[t];
    if (off[P.nt] > sol->cand_cap)
      return fail(SKYOPT_ELIMIT, "candidate table needs %lld entries, capacity %lld",
                  (long long)off[P.nt], (long long)sol->cand_cap);
    memcpy(sol->task_cand_offset, off.data(), sizeof(int64_t) * (P.nt + 1));
    if (off[P.nt] > 0) {
      int64_t *d_off = nullptr; SkyoptCandidate *d_tab = nullptr;
      CU(cudaMalloc(&d_off, sizeof(int64_t) * (P.nt + 1)));
      CU(cudaMalloc(&d_tab, sizeof(SkyoptCandidate) * off[P.nt]));
      CU(cudaMemcpyAsync(d_off, off.data(), sizeof(int64_t) * (P.nt + 1), cudaMemcpyHostToDevice, x->stream));
      ExpandOut ex{P.slot_count, P.slot_inst, P.cand_region, P.cand_zone, P.cand_pa, P.cand_pb};
      SolveIn in{P.slots, P.tasks, P.parents, P.tariffs, P.blocked, P.dags, P.slot_off, P.task_off, ex, 0, P.res, P.nres};
      SolveWork w{P.tc_ref, P.tc_slot, P.tc_cloud, P.tc_hourly, P.tc_value, P.dp, P.back};
      table_kernel<<<P.nt, 128, 0, x->stream>>>(in, w, P.task_n, P.nt, d_off, d_tab);
      cudaError_t e = cudaGetLastError();
      if (e == cudaSuccess)
        e = cudaMemcpyAsync(sol->candidates, d_tab, sizeof(SkyoptCandidate) * off[P.nt],
                            cudaMemcpyDeviceToHost, x->stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(x->stream);
      cudaFree(d_off); cudaFree(d_tab);
      if (e != cudaSuccess) return fail(SKYOPT_ECUDA, "candidate table: %s", cudaGetErrorString(e));
    }
  }
  return 0;
}

int fill_stats(Ctx *x, const Plan &P, SkyoptStats *stats, bool solve) {
  if (!stats) return 0;
  memset(stats, 0, sizeof(*stats));
  if (P.ran_fused) {
    // one launch: the step is not split into phases (SKYOPT_TRACE has the
    // in-kernel timeline)
    CU(cudaEventElapsedTime(&stats->scan_kernel_ms, x->ev[1], x->ev[4]));
    stats->scan_ms = stats->scan_kernel_ms;
  } else {
  CU(cudaEventElapsedTime(&stats->scan_ms, x->ev[1], x->ev[2]));
  if (solve) {
    CU(cudaEventElapsedTime(&stats->expand_ms, x->ev[2], x->ev[3]));
    CU(cudaEventElapsedTime(&stats->solve_ms, x->ev[3], x->ev[4]));
  }
  }
  CU(cudaEventElapsedTime(&stats->total_ms, x->ev[0], x->ev[5]));
  stats->scan_launches = (P.fast ? P.n_pieces : P.n_blocks) ? 1 : 0;
  stats->total_launches = stats->scan_launches + ((P.nq && (P.want_finalize || !solve)) ? 1 : 0) +
                          (solve ? (P.fast ? ((P.nt ? 1 : 0) + (P.nd ? 1 : 0))
                                           : ((P.ns ? 1 : 0) + (P.nd ? 2 : 0))) : 0);
  if (P.ran_fused) { stats->scan_launches = 1; stats->total_launches = 1 + ((P.nd && !P.chain_dags) ? 1 : 0); }
  stats->scan_rows = P.scan_rows;
  stats->scan_passes_rows = P.pass_rows;
  stats->scan_blocks = P.fast ? (P.ran_fused ? P.step_grid : P.scan2_grid) : P.n_blocks;
  stats->scan_form = P.fast ? (P.ran_fused ? 4 : 3) : (P.stream ? 1 : (P.queue ? 2 : 0));
  stats->reserved_ = P.fast ? (int32_t)std::min<int64_t>(P.layout_rows, 0x7FFFFFFF) : 0;
  if (!P.ran_fused && (P.fast ? P.n_pieces : P.n_blocks)) CU(cudaEventElapsedTime(&stats->scan_kernel_ms, x->ev[6], x->ev[7]));
  return 0;
}

}  // namespace

extern "C" {

static_assert(sizeof(SkyoptStats) == 56 && offsetof(SkyoptStats, scan_form) == 48, "SkyoptStats ABI");
int skyopt_abi_version(void) { return SKYOPT_ABI_VERSION; }

uint64_t skyopt_price_key(double price) {
  uint64_t b; memcpy(&b, &price, 8);
  return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
const char *skyopt_last_error(void) { return g_error.c_str(); }

int skyopt_device_count(int *count) {
  if (!count) return fail(SKYOPT_EINVAL, "count is NULL");
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) { *count = 0; return fail(SKYOPT_ENODEV, "cudaGetDeviceCount: %s", cudaGetErrorString(e)); }
  *count = n;
  return 0;
}

int skyopt_catalog_create(const SkyoptCatalogDesc *d, int device, SkyoptCatalog **out) {
  NvtxRange nvtx_("skyopt_catalog_create");
  if (!d || !out) return fail(SKYOPT_EINVAL, "NULL argument");
  *out = nullptr;
  if (d->n_rows <= 0 || d->n_rows % kZoneRows != 0) return fail(SKYOPT_EINVAL, "n_rows must be a positive multiple of 128");
  if (d->n_rows > 0x7FFFFFF0ll) return fail(SKYOPT_ELIMIT, "catalog exceeds 2^31 rows");
  if (d->n_clouds <= 0 || d->n_clouds > SKYOPT_MAX_CLOUDS) return fail(SKYOPT_ELIMIT, "1..%d clouds supported", SKYOPT_MAX_CLOUDS);
  if (d->n_acc_keys < 0 || d->n_acc_keys > 32 * SKYOPT_ACC_SET_WORDS)
    return fail(SKYOPT_ELIMIT, "at most %d distinct (accelerator, count) pairs", 32 * SKYOPT_ACC_SET_WORDS);
  if (!d->price || !d->spot_price || !d->vcpus || !d->mem || !d->acc_key || !d->region_id ||
      !d->zone_id || !d->flags || !d->inst_id || !d->cloud_row_offsets || !d->cloud_inst_offsets ||
      !d->cloud_region_offsets || !d->cloud_n_zones || !d->region_is_us || !d->inst_row_offsets ||
      !d->inst_rows || !d->acc_row_offsets || !d->acc_rows || !d->inst_acc_key || !d->zone_map)
    return fail(SKYOPT_EINVAL, "a required column pointer is NULL");
  if (d->cloud_row_offsets[0] != 0 || d->cloud_row_offsets[d->n_clouds] != d->n_rows)
    return fail(SKYOPT_EINVAL, "cloud_row_offsets must span [0, n_rows]");
  for (int c = 0; c < d->n_clouds; ++c)
    if (d->cloud_row_offsets[c] % kZoneRows != 0 || d->cloud_row_offsets[c + 1] < d->cloud_row_offsets[c])
      return fail(SKYOPT_EINVAL, "cloud %d row range must be 128-row aligned", c);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
    return fail(SKYOPT_ENODEV, "no CUDA device available; libskyopt has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(SKYOPT_EINVAL, "device %d out of range (%d devices)", device, ndev);
  CU(cudaSetDevice(device));
  SkyoptCatalog *c = new (std::nothrow) SkyoptCatalog();
  if (!c) return fail(SKYOPT_ENOMEM, "out of host memory");
  c->device = device;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) c->sm_count = prop.multiProcessorCount;

  const size_t n = (size_t)d->n_rows;
  const size_t slack = kStreamTile;  // one tile of over-read
  int rc = 0;
  CatDev &v = c->dev;
  v.n_rows = d->n_rows;
  v.n_clouds = d->n_clouds; v.n_inst = d->n_inst; v.n_acc_keys = d->n_acc_keys; v.n_regions = d->n_regions;
  const size_t n_inst_rows = (size_t)d->inst_row_offsets[d->n_inst];
  const size_t n_acc_rows = (size_t)d->acc_row_offsets[d->n_acc_keys];
  rc = rc ? rc : upload(c, d->price, n, slack, &v.price);
  rc = rc ? rc : upload(c, d->spot_price, n, slack, &v.spot);
  rc = rc ? rc : upload(c, d->vcpus, n, slack, &v.vcpus);
  rc = rc ? rc : upload(c, d->mem, n, slack, &v.mem);
  if (d->disk_total) rc = rc ? rc : upload(c, d->disk_total, n, slack, &v.disk_total);
  rc = rc ? rc : upload(c, d->acc_key, n, slack, &v.acc_key, 0xFF);
  rc = rc ? rc : upload(c, d->region_id, n, slack, &v.region_id);
  rc = rc ? rc : upload(c, d->zone_id, n, slack, &v.zone_id, 0xFF);
  rc = rc ? rc : upload(c, d->flags, n, slack, &v.flags);
  rc = rc ? rc : upload(c, d->inst_id, n, slack, &v.inst_id, 0xFF);
  rc = rc ? rc : upload(c, d->cloud_row_offsets, (size_t)d->n_clouds + 1, 0, &v.cloud_row_offsets);
  rc = rc ? rc : upload(c, d->cloud_inst_offsets, (size_t)d->n_clouds + 1, 0, &v.cloud_inst_offsets);
  rc = rc ? rc : upload(c, d->cloud_region_offsets, (size_t)d->n_clouds + 1, 0, &v.cloud_region_offsets);
  rc = rc ? rc : upload(c, d->cloud_n_zones, (size_t)d->n_clouds, 0, &v.cloud_n_zones);
  rc = rc ? rc : upload(c, d->region_is_us, (size_t)std::max(d->n_regions, 1), 0, &v.region_is_us);
  rc = rc ? rc : upload(c, d->inst_row_offsets, (size_t)d->n_inst + 1, 0, &v.inst_row_offsets);
  rc = rc ? rc : upload(c, d->inst_rows, n_inst_rows, 1, &v.inst_rows);
  rc = rc ? rc : upload(c, d->acc_row_offsets, (size_t)d->n_acc_keys + 1, 0, &v.acc_row_offsets);
  rc = rc ? rc : upload(c, d->acc_rows, n_acc_rows, 1, &v.acc_rows);
  rc = rc ? rc : upload(c, d->inst_acc_key, (size_t)std::max(d->n_inst, 1), 0, &v.inst_acc_key, 0xFF);
  static_assert(sizeof(SkyoptZone) == sizeof(RowSummary), "zone map ABI");
  rc = rc ? rc : upload(c, reinterpret_cast<const RowSummary *>(d->zone_map), n / kZoneRows,
                        kStreamTile / kZoneRows + 1, &v.zone_map);
  if (rc) { skyopt_catalog_destroy(c); return rc; }

  c->flag_density.assign(d->n_clouds, std::array<float, 256>{});
  for (int cl = 0; cl < d->n_clouds; ++cl) {
    const int64_t z0 = d->cloud_row_offsets[cl] / kZoneRows, z1 = d->cloud_row_offsets[cl + 1] / kZoneRows;
    std::array<int64_t, 256> exact{};  // chunks per exact flag byte
    for (int64_t z = z0; z < z1; ++z) exact[d->zone_map[z].flags_or & 0xFFu]++;
    for (int m = 0; m < 256; ++m) {
      int64_t n = 0;
      for (int f = 0; f < 256; ++f) if ((f & m) == m) n += exact[f];
      c->flag_density[cl][m] = z1 > z0 ? (float)((double)n / (double)(z1 - z0)) : 0.f;
    }
  }
  {
    std::vector<int32_t> tile_list;
    for (int r = 0; r < 3; ++r) {
      const int cpt = 2 << r;  // 128-row chunks per tile
      c->tile_class[r].assign(d->n_clouds, {});
      for (int cl = 0; cl < d->n_clouds; ++cl) {
        const int64_t z0 = d->cloud_row_offsets[cl] / kZoneRows, z1 = d->cloud_row_offsets[cl + 1] / kZoneRows;
        const int n_tiles = (int)((z1 - z0 + cpt - 1) / cpt);
        std::vector<int32_t> members[2];
        std::array<int64_t, 256> exact[2] = {};
        int64_t chunks[2] = {0, 0};
        for (int t = 0; t < n_tiles; ++t) {
          int with_default = 0, n = 0;
          for (int64_t z = z0 + (int64_t)t * cpt; z < std::min<int64_t>(z1, z0 + (int64_t)(t + 1) * cpt); ++z, ++n)
            with_default += (d->zone_map[z].flags_or & SKYOPT_F_DEFAULT_FAMILY) ? 1 : 0;
          const int k = (with_default * 4 >= n) ? 1 : 0;
          members[k].push_back(t);
          for (int64_t z = z0 + (int64_t)t * cpt; z < std::min<int64_t>(z1, z0 + (int64_t)(t + 1) * cpt); ++z)
            exact[k][d->zone_map[z].flags_or & 0xFFu]++;
          chunks[k] += n;
        }
        for (int k = 0; k < 2; ++k) {
          SkyoptCatalog::TileClass &tc = c->tile_class[r][cl][k];
          tc.n_tiles = (int)members[k].size();
          if (tc.n_tiles > 0) {
            tc.tile0 = members[k].front();
            if (members[k].back() - members[k].front() + 1 != tc.n_tiles) {
              tc.list0 = (int)tile_list.size();
              tile_list.insert(tile_list.end(), members[k].begin(), members[k].end());
            }
          }
          for (int m = 0; m < 256; ++m) {
            int64_t n = 0;
            for (int f = 0; f < 256; ++f) if ((f & m) == m) n += exact[k][f];
            tc.density[m] = chunks[k] ? (float)((double)n / (double)chunks[k]) : 0.f;
          }
        }
      }
    }
    if (tile_list.empty()) tile_list.push_back(0);
    rc = upload(c, tile_list.data(), tile_list.size(), 0, &c->d_tile_list);
    if (rc) { skyopt_catalog_destroy(c); return rc; }
  }
  c->cloud_row_offsets.assign(d->cloud_row_offsets, d->cloud_row_offsets + d->n_clouds + 1);
  c->cloud_inst_offsets.assign(d->cloud_inst_offsets, d->cloud_inst_offsets + d->n_clouds + 1);
  c->cloud_region_offsets.assign(d->cloud_region_offsets, d->cloud_region_offsets + d->n_clouds + 1);
  c->cloud_n_zones.assign(d->cloud_n_zones, d->cloud_n_zones + d->n_clouds);
  // Expand capacity per cloud: largest instance-type group, or all
  // accelerator-only rows of one key.
  c->cloud_group_cap.assign(d->n_clouds, 1);
  int max_group = 1;
  for (int cl = 0; cl < d->n_clouds; ++cl) {
    int cap = 1;
    for (int i = d->cloud_inst_offsets[cl]; i < d->cloud_inst_offsets[cl + 1]; ++i)
      cap = std::max(cap, d->inst_row_offsets[i + 1] - d->inst_row_offsets[i]);
    c->cloud_group_cap[cl] = cap;
    c->max_regions = std::max(c->max_regions, d->cloud_region_offsets[cl + 1] - d->cloud_region_offsets[cl]);
    c->max_zones = std::max(c->max_zones, d->cloud_n_zones[cl]);
  }
  // accelerator groups may span clouds in the CSR; bound them by the group
  for (int k = 0; k < d->n_acc_keys; ++k) {
    const int rows = d->acc_row_offsets[k + 1] - d->acc_row_offsets[k];
    if (!rows) continue;
    // an exact accelerator set may union a few keys (case variants): x4 slack
    for (int cl = 0; cl < d->n_clouds; ++cl) {
      bool in_cloud = false;
      for (int i = d->acc_row_offsets[k]; i < d->acc_row_offsets[k + 1] && !in_cloud; ++i)
        in_cloud = d->acc_rows[i] >= d->cloud_row_offsets[cl] && d->acc_rows[i] < d->cloud_row_offsets[cl + 1];
      if (in_cloud) c->cloud_group_cap[cl] = std::max(c->cloud_group_cap[cl], rows);
    }
  }
  for (int cl = 0; cl < d->n_clouds; ++cl) max_group = std::max(max_group, c->cloud_group_cap[cl]);
  if (max_group > SKYOPT_MAX_GROUP_ROWS) {
    skyopt_catalog_destroy(c);
    return fail(SKYOPT_ELIMIT, "an instance type has %d rows; the limit is %d", max_group, SKYOPT_MAX_GROUP_ROWS);
  }
  c->sort_n = std::max(2, next_pow2(max_group));
  for (int cl = 0; cl < d->n_clouds; ++cl) c->cloud_group_cap[cl] = c->sort_n;  // sorted output is written sparsely
  const size_t smem = (size_t)c->sort_n * 16 + (size_t)c->max_zones * 8 + (size_t)c->max_regions * 4;
  if (smem > 200 * 1024) { skyopt_catalog_destroy(c); return fail(SKYOPT_ELIMIT, "expand needs %zu B of shared memory", smem); }
  // The attribute is per function, not per catalog: only ever raise it.
  static std::mutex attr_mu;
  static size_t attr_expand = 48 * 1024;
  cudaError_t e = cudaSuccess;
  {
    std::lock_guard<std::mutex> g(attr_mu);
    if (smem > attr_expand) {
      e = cudaFuncSetAttribute(expand_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e == cudaSuccess) attr_expand = smem;
    }
  }
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(scan_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)(kStreamStages * sizeof(StreamStage)));
  if (e != cudaSuccess) { skyopt_catalog_destroy(c); return fail(SKYOPT_ECUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e)); }
  if (const char *mode = getenv("SKYOPT_SCAN_MODE")) {
    if (!strcmp(mode, "tile")) c->scan_mode = 1;
    else if (!strcmp(mode, "stream")) c->scan_mode = 2;
    else if (!strcmp(mode, "stream3")) c->scan_mode = 3;
    else if (!strcmp(mode, "queue")) c->scan_mode = 4;
    else if (!strcmp(mode, "queue32")) c->scan_mode = 5;
    else if (!strcmp(mode, "fast")) c->scan_mode = 6;
    else if (!strcmp(mode, "fast-noprune")) { c->scan_mode = 6; c->noprune = true; }
    else if (!strcmp(mode, "fast-split")) { c->scan_mode = 6; c->split = true; }
    else if (!strcmp(mode, "fast-split-noprune")) { c->scan_mode = 6; c->split = true; c->noprune = true; }
  }
  rc = build_fast(c, d);
  if (rc) { skyopt_catalog_destroy(c); return rc; }
  if (c->fast_ok) {
    int coop = 0;
    if (cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device) == cudaSuccess) c->coop = coop != 0;
    e = cudaFuncSetAttribute(step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(place_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(PlaceSmem));
    if (e == cudaSuccess)
    e = cudaFuncSetAttribute(scan2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
    if (e != cudaSuccess) { skyopt_catalog_destroy(c); return fail(SKYOPT_ECUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e)); }
  }
  CU(cudaDeviceSynchronize());
  *out = c;
  return 0;
}

int skyopt_catalog_destroy(SkyoptCatalog *c) {
  if (!c) return 0;
  cudaSetDevice(c->device);
  for (Ctx *x : c->free_ctx) {
    if (x->stream) cudaStreamDestroy(x->stream);
    for (auto &e : x->ev) if (e) cudaEventDestroy(e);
    if (x->dbuf) cudaFree(x->dbuf);
    if (x->hbuf) cudaFreeHost(x->hbuf);
    if (x->flush) cudaFree(x->flush);
    if (x->trace) cudaFree(x->trace);
    if (x->sync) cudaFree(x->sync);
    delete x;
  }
  for (void *p : c->allocs) cudaFree(p);
  delete c;
  return 0;
}

int skyopt_catalog_set_scan_mode(SkyoptCatalog *c, int mode) {
  if (!c || mode < 0 || mode > 9)
    return fail(SKYOPT_EINVAL, "scan mode must be 0 (auto), 1 (tile), 2 (stream), 3 (stream, 3 tiles per block), "
                               "4 (queue), 5 (queue, 32 tiles per block), 6 (class-table scan, one fused launch), "
                               "7 (6 without pruning), 8 (6 as separate launches) or 9 (8 without pruning)");
  if (mode >= 6 && !c->fast_ok) return fail(SKYOPT_ELIMIT, "the class-table scan is not available for this catalog");
  c->noprune = mode == 7 || mode == 9;
  c->split = mode == 8 || mode == 9;
  c->scan_mode = mode >= 6 ? 6 : mode;
  return 0;
}

int skyopt_catalog_bytes(const SkyoptCatalog *c, int64_t *device_bytes, int64_t *row_bytes) {
  if (!c) return fail(SKYOPT_EINVAL, "NULL catalog");
  if (device_bytes) *device_bytes = c->device_bytes;
  // bytes the scan streams per row and pass: one price column, vCPUs,
  // MemoryGiB (f64) + acc_key, region, zone, flags (u16)
  if (row_bytes) *row_bytes = 3 * 8 + 4 * 2;
  return 0;
}

int skyopt_list_offerings(SkyoptCatalog *cat, int cloud, int by_acc_key,
                          const int32_t *group_ids, int n_groups,
                          const uint32_t *region_mask, int per_region,
                          int32_t *out_rows) {
  NvtxRange nvtx_("skyopt_list_offerings");
  if (!cat || !group_ids || !out_rows || n_groups <= 0) return fail(SKYOPT_EINVAL, "bad arguments");
  if (cloud < 0 || cloud >= cat->dev.n_clouds) return fail(SKYOPT_EINVAL, "cloud %d out of range", cloud);
  const int n_max = by_acc_key ? cat->dev.n_acc_keys : cat->dev.n_inst;
  for (int i = 0; i < n_groups; ++i)
    if (group_ids[i] < 0 || group_ids[i] >= n_max) return fail(SKYOPT_EINVAL, "group %d: id %d out of range", i, group_ids[i]);
  const int n_regions = cat->cloud_region_offsets[cloud + 1] - cat->cloud_region_offsets[cloud];
  const int slots = per_region ? std::max(n_regions, 1) : 1;
  const size_t smem = (size_t)slots * 20 + 8;
  if (smem > 48 * 1024) return fail(SKYOPT_ELIMIT, "cloud has too many regions (%d)", n_regions);
  CU(cudaSetDevice(cat->device));
  Ctx *x = nullptr;
  int rc = acquire(cat, &x);
  if (rc) return rc;
  int32_t *d_ids = nullptr, *d_out = nullptr; uint32_t *d_mask = nullptr;
  const int mask_words = (std::max(n_regions, 1) + 31) / 32;
  auto body = [&]() -> int {
    cudaStream_t st = x->stream;
    CU(cudaMalloc(&d_ids, sizeof(int32_t) * (size_t)n_groups));
    CU(cudaMalloc(&d_out, sizeof(int32_t) * (size_t)n_groups * slots));
    CU(cudaMemcpyAsync(d_ids, group_ids, sizeof(int32_t) * (size_t)n_groups, cudaMemcpyHostToDevice, st));
    if (region_mask) {
      CU(cudaMalloc(&d_mask, sizeof(uint32_t) * (size_t)mask_words));
      CU(cudaMemcpyAsync(d_mask, region_mask, sizeof(uint32_t) * (size_t)mask_words, cudaMemcpyHostToDevice, st));
    }
    offer_kernel<<<n_groups, 128, smem, st>>>(cat->dev, cloud, by_acc_key ? 1 : 0, d_ids, d_mask,
                                              per_region ? 1 : 0, std::max(n_regions, 1), d_out);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(out_rows, d_out, sizeof(int32_t) * (size_t)n_groups * slots, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return 0;
  };
  rc = body();
  if (rc) cudaStreamSynchronize(x->stream);
  if (d_ids) cudaFree(d_ids);
  if (d_out) cudaFree(d_out);
  if (d_mask) cudaFree(d_mask);
  release(cat, x);
  return rc;
}

int skyopt_scan(SkyoptCatalog *cat, const SkyoptQuery *queries, int n_queries,
                const uint32_t *acc_sets, int n_acc_sets, SkyoptScanResult *results,
                int32_t *list_ids, double *list_prices, int list_cap,
                int32_t *fuzzy_keys, double *fuzzy_prices, int fuzzy_cap,
                SkyoptStats *stats) {
  NvtxRange nvtx_("skyopt_scan");
  if (!cat || !queries || !results || n_queries <= 0) return fail(SKYOPT_EINVAL, "bad arguments");
  if (list_cap > 2048 || fuzzy_cap > 2048) return fail(SKYOPT_ELIMIT, "list capacity is limited to 2048 entries");
  SkyoptProblem pb{};
  pb.queries = queries; pb.n_queries = n_queries; pb.acc_sets = acc_sets; pb.n_acc_sets = n_acc_sets;
  int rc = validate_problem(cat, &pb);
  if (rc) return rc;
  CU(cudaSetDevice(cat->device));
  Ctx *x = nullptr;
  if ((rc = acquire(cat, &x))) return rc;
  Plan P;
  rc = build_plan(cat, &pb, x, P);
  const bool want_list = list_ids && list_prices && list_cap > 0;
  const bool want_fuzzy = fuzzy_keys && fuzzy_prices && fuzzy_cap > 0;
  int32_t *d_ids = nullptr, *d_cnt = nullptr; double *d_pr = nullptr;
  auto body = [&]() -> int {
    if (rc) return rc;
    cudaStream_t st = x->stream;
    CU(cudaEventRecord(x->ev[0], st));
    CU(cudaMemcpyAsync(x->dbuf, x->hbuf, P.in_bytes, cudaMemcpyHostToDevice, st));
    int r = enqueue_kernels(cat, x, P, false);
    if (r) return r;
    CU(cudaMemcpyAsync(x->hbuf, x->dbuf + P.out_off, P.out_bytes, cudaMemcpyDeviceToHost, st));
    CU(cudaEventRecord(x->ev[5], st));
    CU(cudaStreamSynchronize(st));
    Plan H;
    carve_output_host(P, x->hbuf, H);
    fill_scan_results(cat, P, H, results);
    for (int kind = 0; kind < 2; ++kind) {
      const bool want = kind == 0 ? want_list : want_fuzzy;
      if (!want) continue;
      const int cap = kind == 0 ? list_cap : fuzzy_cap;
      const int n_entries_max = kind == 0 ? cat->dev.n_inst : cat->dev.n_acc_keys;
      const int sort_n = std::min(2048, std::max(2, next_pow2(std::max(n_entries_max, cap))));
      CU(cudaMalloc(&d_ids, sizeof(int32_t) * (size_t)n_queries * cap));
      CU(cudaMalloc(&d_pr, sizeof(double) * (size_t)n_queries * cap));
      CU(cudaMalloc(&d_cnt, sizeof(int32_t) * (size_t)n_queries));
      list_kernel<<<n_queries, 256, (size_t)sort_n * 16, st>>>(
          cat->dev, P.queries, kind, kind == 0 ? P.list_base : P.fuzzy_base,
          kind == 0 ? P.list_min : P.fuzzy_min, cap, sort_n, d_ids, d_pr, d_cnt);
      CU(cudaGetLastError());
      std::vector<int32_t> cnt(n_queries);
      CU(cudaMemcpyAsync(kind == 0 ? list_ids : fuzzy_keys, d_ids, sizeof(int32_t) * (size_t)n_queries * cap, cudaMemcpyDeviceToHost, st));
      CU(cudaMemcpyAsync(kind == 0 ? list_prices : fuzzy_prices, d_pr, sizeof(double) * (size_t)n_queries * cap, cudaMemcpyDeviceToHost, st));
      CU(cudaMemcpyAsync(cnt.data(), d_cnt, sizeof(int32_t) * (size_t)n_queries, cudaMemcpyDeviceToHost, st));
      CU(cudaStreamSynchronize(st));
      for (int i = 0; i < n_queries; ++i) (kind == 0 ? results[i].n_list : results[i].n_fuzzy) = cnt[i];
      cudaFree(d_ids); cudaFree(d_pr); cudaFree(d_cnt);
      d_ids = nullptr; d_pr = nullptr; d_cnt = nullptr;
    }
    return fill_stats(x, P, stats, false);
  };
  rc = body();
  if (d_ids) cudaFree(d_ids);
  if (d_pr) cudaFree(d_pr);
  if (d_cnt) cudaFree(d_cnt);
  if (rc) cudaStreamSynchronize(x->stream);
  release(cat, x);
  return rc;
}

int skyopt_optimize(SkyoptCatalog *cat, const SkyoptProblem *pb, SkyoptSolution *sol,
                    SkyoptStats *stats) {
  NvtxRange nvtx_("skyopt_optimize");
  if (!cat || !pb || !sol) return fail(SKYOPT_EINVAL, "NULL argument");
  if (pb->n_dags <= 0 || pb->n_tasks <= 0 || pb->n_slots <= 0)
    return fail(SKYOPT_EINVAL, "empty problem");
  int rc = validate_problem(cat, pb);
  if (rc) return rc;
  CU(cudaSetDevice(cat->device));
  Ctx *x = nullptr;
  if ((rc = acquire(cat, &x))) return rc;
  Plan P;
  auto body = [&]() -> int {
    int r = build_plan(cat, pb, x, P);
    if (r) return r;
    cudaStream_t st = x->stream;
    CU(cudaEventRecord(x->ev[0], st));
    CU(cudaMemcpyAsync(x->dbuf, x->hbuf, P.in_bytes, cudaMemcpyHostToDevice, st));
    P.want_finalize = sol->scan != nullptr;
    if ((r = enqueue_kernels(cat, x, P, true, sol->scan != nullptr))) return r;
    CU(cudaMemcpyAsync(x->hbuf, x->dbuf + P.out_off, P.out_bytes, cudaMemcpyDeviceToHost, st));
    CU(cudaEventRecord(x->ev[5], st));
    CU(cudaStreamSynchronize(st));
    if ((r = copy_solution(cat, x, P, pb, sol))) return r;
    return fill_stats(x, P, stats, true);
  };
  rc = body();
  if (rc) cudaStreamSynchronize(x->stream);
  release(cat, x);
  return rc;
}

struct SkyoptSession {
  SkyoptCatalog *cat = nullptr;
  Ctx *x = nullptr;
  Plan P;
  std::vector<SkyoptDag> dags;       // host copy: task ranges, flags
  SkyoptBlocked *d_blocked = nullptr;
  SkyoptDag *d_dags = nullptr;
  int blocked_cap = 0;
};

int skyopt_session_open(SkyoptCatalog *cat, const SkyoptProblem *pb, SkyoptSolution *sol,
                        SkyoptStats *stats, SkyoptSession **out) {
  NvtxRange nvtx_("skyopt_session_open");
  if (!cat || !pb || !sol || !out) return fail(SKYOPT_EINVAL, "NULL argument");
  *out = nullptr;
  if (pb->n_dags <= 0 || pb->n_tasks <= 0 || pb->n_slots <= 0)
    return fail(SKYOPT_EINVAL, "empty problem");
  int rc = validate_problem(cat, pb);
  if (rc) return rc;
  CU(cudaSetDevice(cat->device));
  SkyoptSession *s = new (std::nothrow) SkyoptSession();
  if (!s) return fail(SKYOPT_ENOMEM, "out of host memory");
  s->cat = cat;
  if ((rc = acquire(cat, &s->x))) { delete s; return rc; }
  Ctx *x = s->x;
  auto body = [&]() -> int {
    int r = build_plan(cat, pb, x, s->P);
    if (r) return r;
    cudaStream_t st = x->stream;
    CU(cudaEventRecord(x->ev[0], st));
    CU(cudaMemcpyAsync(x->dbuf, x->hbuf, s->P.in_bytes, cudaMemcpyHostToDevice, st));
    s->P.want_finalize = sol->scan != nullptr;
    if ((r = enqueue_kernels(cat, x, s->P, true, sol->scan != nullptr))) return r;
    CU(cudaMemcpyAsync(x->hbuf, x->dbuf + s->P.out_off, s->P.out_bytes, cudaMemcpyDeviceToHost, st));
    CU(cudaEventRecord(x->ev[5], st));
    CU(cudaStreamSynchronize(st));
    if ((r = copy_solution(cat, x, s->P, pb, sol))) return r;
    return fill_stats(x, s->P, stats, true);
  };
  rc = body();
  if (rc) {
    cudaStreamSynchronize(x->stream);
    release(cat, x);
    delete s;
    return rc;
  }
  s->dags.assign(pb->dags, pb->dags + pb->n_dags);
  *out = s;
  return 0;
}

int skyopt_session_resolve(SkyoptSession *s, const SkyoptBlocked *blocked, int n_blocked,
                           SkyoptSolution *sol, SkyoptStats *stats) {
  NvtxRange nvtx_("skyopt_session_resolve");
  if (!s || !sol || n_blocked < 0 || (n_blocked > 0 && !blocked)) return fail(SKYOPT_EINVAL, "bad arguments");
  SkyoptCatalog *cat = s->cat;
  Ctx *x = s->x;
  Plan &P = s->P;
  CU(cudaSetDevice(cat->device));
  cudaStream_t st = x->stream;
  if (n_blocked > s->blocked_cap || !s->d_dags) {
    const int cap = std::max(64, 2 * n_blocked);
    SkyoptBlocked *nb = nullptr;
    CU(cudaMalloc(&nb, sizeof(SkyoptBlocked) * (size_t)cap));
    if (s->d_blocked) { CU(cudaStreamSynchronize(st)); cudaFree(s->d_blocked); }
    s->d_blocked = nb; s->blocked_cap = cap;
    if (!s->d_dags) CU(cudaMalloc(&s->d_dags, sizeof(SkyoptDag) * s->dags.size()));
  }
  for (SkyoptDag &d : s->dags) { d.blocked_begin = 0; d.blocked_end = n_blocked; }
  // The copies below read pageable host memory: they are staged before the
  // call returns, and the stream is synchronised further down.
  if (n_blocked) CU(cudaMemcpyAsync(s->d_blocked, blocked, sizeof(SkyoptBlocked) * (size_t)n_blocked, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(s->d_dags, s->dags.data(), sizeof(SkyoptDag) * s->dags.size(), cudaMemcpyHostToDevice, st));
  P.blocked = s->d_blocked; P.dags = s->d_dags;
  CU(cudaEventRecord(x->ev[0], st));
  CU(cudaEventRecord(x->ev[1], st));
  CU(cudaEventRecord(x->ev[6], st)); CU(cudaEventRecord(x->ev[7], st));
  CU(cudaEventRecord(x->ev[2], st));
  CU(cudaEventRecord(x->ev[3], st));
  {
    ExpandOut ex{P.slot_count, P.slot_inst, P.cand_region, P.cand_zone, P.cand_pa, P.cand_pb};
    SolveIn in{P.slots, P.tasks, P.parents, P.tariffs, P.blocked, P.dags, P.slot_off, P.task_off, ex, 0, P.res, P.nres};
    SolveWork w{P.tc_ref, P.tc_slot, P.tc_cloud, P.tc_hourly, P.tc_value, P.dp, P.back};
    SolveOut out{P.chosen, P.chosen_index, P.task_n, P.dagres};
    gather_kernel<<<P.nt, kGatherThreads, 0, st>>>(cat->dev, in, w, P.task_dag, P.task_n);
    CU(cudaGetLastError());
    solve_kernel<<<P.nd, kSolveThreads, 0, st>>>(cat->dev, in, w, out);
    CU(cudaGetLastError());
  }
  CU(cudaEventRecord(x->ev[4], st));
  CU(cudaMemcpyAsync(x->hbuf, x->dbuf + P.out_off, P.out_bytes, cudaMemcpyDeviceToHost, st));
  CU(cudaEventRecord(x->ev[5], st));
  CU(cudaStreamSynchronize(st));
  SkyoptProblem pb{};
  pb.dags = s->dags.data(); pb.n_dags = (int)s->dags.size();
  int rc = copy_solution(cat, x, P, &pb, sol);
  if (rc) return rc;
  rc = fill_stats(x, P, stats, true);
  if (stats && !rc) {
    // nothing was scanned or expanded this time
    stats->scan_launches = 0; stats->total_launches = 2;
    stats->scan_rows = 0; stats->scan_passes_rows = 0; stats->scan_blocks = 0;
    stats->scan_form = 0; stats->reserved_ = 0;
    stats->scan_kernel_ms = 0.f;
  }
  return rc;
}

void skyopt_session_close(SkyoptSession *s) {
  if (!s) return;
  cudaSetDevice(s->cat->device);
  cudaStreamSynchronize(s->x->stream);
  if (s->d_blocked) cudaFree(s->d_blocked);
  if (s->d_dags) cudaFree(s->d_dags);
  release(s->cat, s->x);
  delete s;
}

int skyopt_solve_tables(SkyoptCatalog *cat, const double *values, const int32_t *clouds,
                        const int64_t *task_offsets, const SkyoptTask *tasks, int n_tasks,
                        const int32_t *parents, int n_parents, const double *tariffs,
                        int n_tariffs, const SkyoptDag *dags, int n_dags,
                        int32_t *chosen_index, SkyoptDagResult *results) {
  NvtxRange nvtx_("skyopt_solve_tables");
  if (!cat || !values || !clouds || !task_offsets || !tasks || !dags || !chosen_index || !results ||
      n_tasks <= 0 || n_dags <= 0)
    return fail(SKYOPT_EINVAL, "bad arguments");
  const int C = cat->dev.n_clouds;
  SkyoptProblem pb{};
  pb.tasks = tasks; pb.n_tasks = n_tasks; pb.parents = parents; pb.n_parents = n_parents;
  pb.tariffs = tariffs; pb.n_tariffs = n_tariffs; pb.dags = dags; pb.n_dags = n_dags;
  // reuse the structural checks (slot ranges are irrelevant here)
  std::vector<SkyoptTask> tk(tasks, tasks + n_tasks);
  for (auto &t : tk) { t.slot_begin = 0; t.slot_end = 0; }
  pb.tasks = tk.data();
  int rc = validate_problem(cat, &pb);
  if (rc) return rc;
  const int64_t total = task_offsets[n_tasks];
  if (task_offsets[0] != 0 || total < 0) return fail(SKYOPT_EINVAL, "bad task_offsets");
  for (int t = 0; t < n_tasks; ++t)
    if (task_offsets[t + 1] < task_offsets[t]) return fail(SKYOPT_EINVAL, "bad task_offsets");
  for (int64_t i = 0; i < total; ++i)
    if (clouds[i] < 0 || clouds[i] >= C) return fail(SKYOPT_EINVAL, "candidate %lld: bad cloud", (long long)i);
  CU(cudaSetDevice(cat->device));
  Ctx *x = nullptr;
  if ((rc = acquire(cat, &x))) return rc;
  auto body = [&]() -> int {
    Carver sizing(nullptr);
    auto carve = [&](Carver &c, double *&d_val, int32_t *&d_cl, int64_t *&d_off, SkyoptTask *&d_tasks,
                     int32_t *&d_par, double *&d_tar, SkyoptDag *&d_dags, int32_t *&d_tn,
                     double *&d_dp, int32_t *&d_back, int32_t *&d_idx, SkyoptDagResult *&d_res) {
      d_val = c.take<double>(total); d_cl = c.take<int32_t>(total);
      d_off = c.take<int64_t>(n_tasks + 1); d_tasks = c.take<SkyoptTask>(n_tasks);
      d_par = c.take<int32_t>(n_parents); d_tar = c.take<double>(n_tariffs);
      d_dags = c.take<SkyoptDag>(n_dags); d_tn = c.take<int32_t>(n_tasks);
      d_dp = c.take<double>(total); d_back = c.take<int32_t>(total);
      d_idx = c.take<int32_t>(n_tasks); d_res = c.take<SkyoptDagResult>(n_dags);
    };
    double *v, *tar, *dp; int32_t *cl, *par, *tn, *back, *idx; int64_t *off;
    SkyoptTask *dt; SkyoptDag *dd; SkyoptDagResult *res;
    carve(sizing, v, cl, off, dt, par, tar, dd, tn, dp, back, idx, res);
    int r = ensure(x, align_up(sizing.off), 256);
    if (r) return r;
    Carver d(x->dbuf);
    carve(d, v, cl, off, dt, par, tar, dd, tn, dp, back, idx, res);
    cudaStream_t st = x->stream;
    std::vector<int32_t> counts(n_tasks);
    for (int t = 0; t < n_tasks; ++t) counts[t] = (int32_t)(task_offsets[t + 1] - task_offsets[t]);
    CU(cudaMemcpyAsync(v, values, sizeof(double) * total, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(cl, clouds, sizeof(int32_t) * total, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(off, task_offsets, sizeof(int64_t) * (n_tasks + 1), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(dt, tk.data(), sizeof(SkyoptTask) * n_tasks, cudaMemcpyHostToDevice, st));
    if (n_parents) CU(cudaMemcpyAsync(par, parents, sizeof(int32_t) * n_parents, cudaMemcpyHostToDevice, st));
    if (n_tariffs) CU(cudaMemcpyAsync(tar, tariffs, sizeof(double) * n_tariffs, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(dd, dags, sizeof(SkyoptDag) * n_dags, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(tn, counts.data(), sizeof(int32_t) * n_tasks, cudaMemcpyHostToDevice, st));
    SolveIn in{nullptr, dt, par, tar, nullptr, dd, nullptr, off, ExpandOut{}, 1};
    SolveWork w{nullptr, nullptr, cl, nullptr, v, dp, back};
    SolveOut out{nullptr, idx, tn, res};
    solve_kernel<<<n_dags, kSolveThreads, 0, st>>>(cat->dev, in, w, out);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(chosen_index, idx, sizeof(int32_t) * n_tasks, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(results, res, sizeof(SkyoptDagResult) * n_dags, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    for (int d2 = 0; d2 < n_dags; ++d2)
      if (results[d2].status != 0)
        for (int t = dags[d2].task_begin; t < dags[d2].task_end; ++t) chosen_index[t] = -1;
    return 0;
  };
  rc = body();
  if (rc) cudaStreamSynchronize(x->stream);
  release(cat, x);
  return rc;
}

int skyopt_optimize_timed(SkyoptCatalog *cat, const SkyoptProblem *pb, SkyoptSolution *sol,
                          int iters, int flush_l2, float *iter_ms, float *scan_ms,
                          SkyoptStats *stats) {
  if (!cat || !pb || !sol || iters <= 0 || !iter_ms) return fail(SKYOPT_EINVAL, "bad arguments");
  int rc = validate_problem(cat, pb);
  if (rc) return rc;
  CU(cudaSetDevice(cat->device));
  Ctx *x = nullptr;
  if ((rc = acquire(cat, &x))) return rc;
  Plan P;
  auto body = [&]() -> int {
    int r = build_plan(cat, pb, x, P);
    if (r) return r;
    cudaStream_t st = x->stream;
    const size_t flush_words = (size_t)192 << 20 >> 2;  // 192 MB > 126 MB L2
    if (flush_l2 && !x->flush) {
      CU(cudaMalloc(&x->flush, flush_words * 8));  // second half: read pass
      CU(cudaMemset(x->flush + flush_words, 0, flush_words * 4));
      x->flush_words = flush_words;
    }
    const char *trace_path = getenv("SKYOPT_TRACE");
    const size_t trace_words = (size_t)3 * kTraceBlocks * kTraceSlots;
    if (trace_path && !x->trace) CU(cudaMalloc(&x->trace, trace_words * 8));
    if (!trace_path && x->trace) { cudaFree(x->trace); x->trace = nullptr; }
    CU(cudaEventRecord(x->ev[0], st));
    CU(cudaMemcpyAsync(x->dbuf, x->hbuf, P.in_bytes, cudaMemcpyHostToDevice, st));
    P.want_finalize = sol->scan != nullptr;
    for (int it = 0; it < iters; ++it) {
      if (x->trace) CU(cudaMemsetAsync(x->trace, 0, trace_words * 8, st));
      if (flush_l2) {
        flush_kernel<<<cat->sm_count * 8, 256, 0, st>>>(x->flush, (int64_t)x->flush_words, (uint32_t)it);
        CU(cudaGetLastError());
        static const bool read_pass = [] { const char *e = getenv("SKYOPT_FLUSH"); return e && !strcmp(e, "read"); }();
        if (read_pass) {
          flush_read_kernel<<<cat->sm_count * 8, 256, 0, st>>>(x->flush + x->flush_words, (int64_t)x->flush_words, x->flush);
          CU(cudaGetLastError());
        }
      }
      P.fresh_inputs = false;  // the timed region resets the scan results itself
      if ((r = enqueue_kernels(cat, x, P, true, sol->scan != nullptr))) return r;
      CU(cudaStreamSynchronize(st));
      CU(cudaEventElapsedTime(&iter_ms[it], x->ev[1], x->ev[4]));
      if (scan_ms && !P.ran_fused && (P.fast ? P.n_pieces : P.n_blocks)) CU(cudaEventElapsedTime(&scan_ms[it], x->ev[6], x->ev[7]));
      if (scan_ms && P.ran_fused) scan_ms[it] = iter_ms[it];
    }
    if (x->trace) {
      // the last iteration's per-block timeline (tools/trace2.py reads it)
      std::vector<unsigned long long> h(trace_words);
      CU(cudaMemcpy(h.data(), x->trace, trace_words * 8, cudaMemcpyDeviceToHost));
      // one file per timing loop of the process: <path>, <path>.1, <path>.2, ...
      static int trace_calls = 0;
      std::string path = trace_path;
      if (trace_calls) path += "." + std::to_string(trace_calls);
      ++trace_calls;
      if (FILE *f = fopen(path.c_str(), "wb")) { fwrite(h.data(), 8, h.size(), f); fclose(f); }
    }
    CU(cudaMemcpyAsync(x->hbuf, x->dbuf + P.out_off, P.out_bytes, cudaMemcpyDeviceToHost, st));
    CU(cudaEventRecord(x->ev[5], st));
    CU(cudaStreamSynchronize(st));
    if ((r = copy_solution(cat, x, P, pb, sol))) return r;
    return fill_stats(x, P, stats, true);
  };
  rc = body();
  if (rc) cudaStreamSynchronize(x->stream);
  release(cat, x);
  return rc;
}

}  // extern "C"
