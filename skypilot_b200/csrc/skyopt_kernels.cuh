// skyopt_kernels.cuh -- sm_100a kernels of the placement-optimizer hot path.
//
// K1 scan_kernel      Resources-constraint filter + per-query argmin over the
//                     SoA catalog (reference sky/catalog/common.py:518-569,
//                     :641-694). HBM-bound: one pass over 32 B/row streams the
//                     rows once for up to 32 fused queries whose constraint
//                     vectors sit in shared memory.
// K1b finalize_kernel per-query reduction of the per-tile partials.
// K1c list_kernel     sorted (instance type, min price) / fuzzy tables.
// K2 expand_kernel    region/zone expansion of the winning instance type,
//                     ordering and per-candidate hourly price
//                     (common.py:793-809, :360-400; resources_utils.py:454-502;
//                     gcp.py:281-331; gcp_catalog.py:424-442).
// K3 solve_kernel     blocked filter, cost, egress and chain DP / exact DAG
//                     search (optimizer.py:196-236, :343-357, :429-487,
//                     :490-637; resources.py:1938-1961).
//
// No tensor cores: this path is scan / filter / reduce (BASELINE.json).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "skyopt.h"
#include "skyopt_reserve.cuh"

namespace skyopt {

constexpr int kScanThreads = 256;
#ifndef SKYOPT_SCAN_BLOCKS_PER_SM
#define SKYOPT_SCAN_BLOCKS_PER_SM 3
#endif
constexpr int kScanBlocksPerSM = SKYOPT_SCAN_BLOCKS_PER_SM;
constexpr int kQChunk = 32;           // queries fused per pass
constexpr uint64_t kKeyNone = 0xFFFFFFFFFFFFFFFFull;
constexpr uint64_t kKeyNaN = 0xFFFFFFFFFFFFFFF0ull;  // after every real price
constexpr uint32_t kRowNone = 0xFFFFFFFFu;

struct CatDev {
  int64_t n_rows;
  const double *price, *spot, *vcpus, *mem, *disk_total;
  const uint16_t *acc_key, *region_id, *zone_id, *flags;
  const int32_t *inst_id;
  const int32_t *cloud_row_offsets, *cloud_inst_offsets, *cloud_region_offsets;
  const int32_t *cloud_n_zones;
  const uint8_t *region_is_us;
  const int32_t *inst_row_offsets, *inst_rows, *acc_row_offsets, *acc_rows;
  const uint16_t *inst_acc_key;
  const struct RowSummary *zone_map;  // one entry per 128 rows
  int32_t n_clouds, n_inst, n_acc_keys, n_regions;
};

// One (cloud, query-chunk) unit of the scan grid.
struct ScanGroup {
  int32_t row_begin, row_end;
  int32_t q_begin, q_count;  // into q_order
  int32_t block0, n_tiles;   // first block, number of blocks (partials)
  uint32_t need;             // bit0 on-demand column, bit1 spot column
  int32_t tiles_per_block;   // stream kernel: consecutive tiles per block
  int32_t total_tiles;       // stream kernel: tiles of the row range
  int32_t list0;             // first entry of the group's tile list; -1 = the run
  int32_t tile0;             //   of consecutive tiles starting at tile0
  int32_t pad_;
};

struct ScanPartial {
  uint64_t key;
  uint32_t row;
  uint32_t pad_;
};

struct ScanFinal {
  uint64_t key;
  int32_t row;
  int32_t inst;
};

// Total order on prices as unsigned integers (NaN never reaches here).
__host__ __device__ __forceinline__ uint64_t price_key(double p) {
#ifdef __CUDA_ARCH__
  uint64_t b = (uint64_t)__double_as_longlong(p);
#else
  uint64_t b; memcpy(&b, &p, 8);
#endif
  return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double key_price(uint64_t k) {
  uint64_t b = (k & 0x8000000000000000ull) ? (k & 0x7FFFFFFFFFFFFFFFull) : ~k;
  return __longlong_as_double((long long)b);
}

__device__ __forceinline__ bool test_bit(const uint32_t *set, uint32_t k) {
  return (set[k >> 5] >> (k & 31)) & 1u;
}

// Constraint vector of one query as the scan loop wants it: everything that
// is an equality test on small integers (flags, group, region, zone, row
// validity) is folded into one 64-bit (mask, value) pair against the row key
//   key = flags | region << 16 | zone << 32,
// and the vCPU / memory operators become closed intervals.
struct QueryS {
  uint32_t mask_lo, mask_hi, val_lo, val_hi;
  uint32_t qflags;       // SKYOPT_Q_*
  uint32_t flags2;       // flags_require2
  int32_t price_col, cpus_op, mem_op, disk_op;
  int32_t cloud;
  uint32_t req_flags;    // flag bits every matching row carries
  uint32_t sig_lo, sig_hi;  // 64-bit signature of the accelerator keys wanted
  uint32_t grp_bit;      // bit (group % 32) of a fixed-host group query, else 0
  uint32_t pad_;
  double cpu_lo, cpu_hi, mem_lo, mem_hi, cap, disk_size;
};

__host__ __device__ inline QueryS make_query_s(const SkyoptQuery &q) {
  const double kInf = 1.0 / 0.0;
  QueryS s;
  uint64_t mask = (uint64_t)((q.flags_require | SKYOPT_F_VALID) & 0xFFu);
  uint64_t val = mask;
  if (q.group != 0) { mask |= 0xFF00ull; val |= ((uint64_t)(q.group & 0xFF)) << 8; }
  if (q.region_id >= 0) { mask |= 0xFFFFull << 16; val |= ((uint64_t)(q.region_id & 0xFFFF)) << 16; }
  if (q.zone_id >= 0) { mask |= 0xFFFFull << 32; val |= ((uint64_t)(q.zone_id & 0xFFFF)) << 32; }
  s.mask_lo = (uint32_t)mask; s.mask_hi = (uint32_t)(mask >> 32);
  s.val_lo = (uint32_t)val; s.val_hi = (uint32_t)(val >> 32);
  s.qflags = q.qflags; s.flags2 = q.flags_require2;
  s.price_col = q.price_col; s.cpus_op = q.cpus_op; s.mem_op = q.mem_op;
  s.disk_op = q.disk_op; s.cloud = q.cloud;
  s.req_flags = (q.flags_require | SKYOPT_F_VALID) & 0xFFu;
  s.sig_lo = 0xFFFFFFFFu; s.sig_hi = 0xFFFFFFFFu;  // refined while staging the sets
  s.grp_bit = (q.group != 0) ? (1u << (q.group & 31)) : 0u;
  s.pad_ = 0;
  s.cpu_lo = q.cpus; s.cpu_hi = (q.cpus_op == SKYOPT_OP_GE) ? kInf : q.cpus;
  s.mem_lo = q.mem;  s.mem_hi = (q.mem_op == SKYOPT_OP_EQ) ? q.mem : kInf;
  s.cap = q.max_price; s.disk_size = q.disk_size;
  return s;
}

// 128-bit (f64) / 64-bit (u16) vector loads through the read-only path. The
// catalog arrays are 256 B aligned, cloud ranges are padded to 8 rows and the
// arrays carry one tile of slack, so every thread's RPT-row group is aligned
// and in bounds.
template <int RPT>
__device__ __forceinline__ void load_f64(const double *__restrict__ col,
                                         int64_t base, double (&out)[RPT]) {
  if constexpr (RPT == 4) {
    const double2 *p = reinterpret_cast<const double2 *>(col + base);
    double2 a = __ldg(p), b = __ldg(p + 1);
    out[0] = a.x; out[1] = a.y; out[2] = b.x; out[3] = b.y;
  } else if constexpr (RPT == 2) {
    double2 a = __ldg(reinterpret_cast<const double2 *>(col + base));
    out[0] = a.x; out[1] = a.y;
  } else {
    out[0] = __ldg(col + base);
  }
}
template <int RPT>
__device__ __forceinline__ void load_u16(const uint16_t *__restrict__ col,
                                         int64_t base, uint32_t (&out)[RPT]) {
  if constexpr (RPT == 4) {
    uint2 a = __ldg(reinterpret_cast<const uint2 *>(col + base));
    out[0] = a.x & 0xFFFF; out[1] = a.x >> 16;
    out[2] = a.y & 0xFFFF; out[3] = a.y >> 16;
  } else if constexpr (RPT == 2) {
    uint32_t a = __ldg(reinterpret_cast<const uint32_t *>(col + base));
    out[0] = a & 0xFFFF; out[1] = a >> 16;
  } else {
    out[0] = __ldg(col + base);
  }
}

constexpr int kSetStride = SKYOPT_ACC_SET_WORDS + 1;  // + a zero word for "no key"
constexpr int kScanWarps = kScanThreads / 32;

// One query in scan order, exactly as a block stages it: the host lays these
// records out per (cloud, chunk) group, so staging is ONE coalesced copy with
// no dependent look-ups (set indices, partial offsets and signatures are
// resolved on the host).
struct ScanQuery {
  QueryS s;
  int32_t qid;           // index in the caller's query array
  int32_t partial_base;  // first partial of this query
  int64_t list_base;     // into list_min (SKYOPT_Q_LIST)
  int64_t fuzzy_base;    // into fuzzy_min (SKYOPT_Q_FUZZY)
  uint32_t set[2][kSetStride];  // exact / fuzzy accelerator-key bitmasks
};
static_assert(sizeof(ScanQuery) % 16 == 0, "ScanQuery is staged with 16-byte loads");

// What the zone-map test needs of a query (same order as the ScanQuery
// records): a block reads these straight from global memory, one per lane,
// and stages the full records only of the queries that survive for at least
// one of its warps.
struct QueryTest {
  uint32_t req_flags, grp_bit, sig_lo, sig_hi;
  uint32_t qflags, price_col;
  int32_t partial_base;
  uint32_t pad_;
};
static_assert(sizeof(QueryTest) == 32, "QueryTest is read as two 16-byte words");

// Shared-memory state of one scan block: the staged queries and the per-warp
// running minima.
struct ScanShared {
  ScanQuery q[kQChunk];
  uint64_t wkey[kQChunk][kScanWarps];
  uint32_t wrow[kQChunk][kScanWarps];
  // best price key found so far, one copy per warp: a warp reads and tightens
  // its own (any achieved key is a valid bound; no cross-warp hand-off)
  uint64_t gb[kQChunk][kScanWarps];
  uint32_t sany[kQChunk];
  uint32_t wact[kScanWarps];  // per-warp masks of surviving queries
};

constexpr int kInlineGroups = 32;

struct ScanArgs {
  CatDev cat;
  const ScanQuery *squeries;   // scan order
  const QueryTest *qtests;     // scan order, parallel to squeries
  const ScanGroup *groups;
  int n_groups;
  ScanPartial *partials;
  unsigned long long *list_min;
  unsigned long long *fuzzy_min;
  unsigned long long *gbest;   // [n_queries] in scan order: running best key
  const int32_t *tile_list;    // static tile classes (see SkyoptCatalog::TileClass)
  int32_t *zero_flag;          // cleared by the first block (expand's error flag)
  int n_blocks;                // grid size
  uint32_t perm_mul;           // odd, coprime with n_blocks
  uint32_t debug;              // bit 1: record the per-block timeline (profiling)
  uint32_t trace_vb, trace_warp;  // debug & 4: per-iteration trace of one warp
  uint32_t qsplit;                // queue form: queries per work entry
  unsigned long long *timeline;  // debug & 2: per block {start, staged, scored, end} ns + smid
  int32_t inline_block0[kInlineGroups];    // first block of each group
  ScanGroup inline_groups[kInlineGroups];  // copy of groups[] when it fits
};

// Launch order -> work unit. Expensive tiles (rows that many queries match)
// sit next to each other in the catalog; a multiplicative permutation spreads
// them over the whole launch instead of leaving them to the last wave.
__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void mark(const ScanArgs &a, int slot) {
  if ((a.debug & 2u) && threadIdx.x == 0) {
    a.timeline[(size_t)blockIdx.x * 8 + slot] = global_ns();
    if (slot == 0) {
      unsigned smid;
      asm volatile("mov.u32 %0, %smid;" : "=r"(smid));
      a.timeline[(size_t)blockIdx.x * 8 + 7] = smid;
    }
  }
}

__device__ __forceinline__ int permuted_block(const ScanArgs &a) {
  return (int)(((uint64_t)blockIdx.x * a.perm_mul) % (uint32_t)a.n_blocks);
}

__device__ __forceinline__ ScanGroup find_group(const ScanArgs &a, int b) {
  // blockIdx -> group: groups are sorted by block0. Small tables travel in
  // the kernel parameters (constant bank, no memory round trip): five
  // branch-free halving steps over the first-block table, then one record.
  if (a.n_groups <= kInlineGroups) {
    int idx = 0;
#pragma unroll
    for (int step = kInlineGroups / 2; step >= 1; step >>= 1) {
      const int probe = idx + step;
      if (probe < a.n_groups && a.inline_block0[probe] <= b) idx = probe;
    }
    return a.inline_groups[idx];
  }
  int lo = 0, hi = a.n_groups - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(&a.groups[mid].block0) <= b) lo = mid; else hi = mid - 1;
  }
  return a.groups[lo];
}

// Stage the chunk's queries: one coalesced copy. Ends with a barrier.
__device__ __forceinline__ void stage_queries(const ScanArgs &a, const ScanGroup &G,
                                              ScanShared &S) {
  const int tid = threadIdx.x;
  const int nq = G.q_count;
  // All of a thread's 16-byte loads are issued before the first store, so a
  // full chunk costs one L2 round trip instead of one per loop iteration.
  const uint4 *src = reinterpret_cast<const uint4 *>(a.squeries + G.q_begin);
  uint4 *dst = reinterpret_cast<uint4 *>(S.q);
  const int n16 = nq * (int)(sizeof(ScanQuery) / 16);
  constexpr int kStageLoads =
      (kQChunk * (int)(sizeof(ScanQuery) / 16) + kScanThreads - 1) / kScanThreads;
  uint4 v[kStageLoads];
#pragma unroll
  for (int k = 0; k < kStageLoads; ++k) {
    const int i = tid + k * kScanThreads;
    if (i < n16) v[k] = __ldg(src + i);
  }
#pragma unroll
  for (int k = 0; k < kStageLoads; ++k) {
    const int i = tid + k * kScanThreads;
    if (i < n16) dst[i] = v[k];
  }
  for (int i = tid; i < nq * kScanWarps; i += kScanThreads) {
    S.wkey[i / kScanWarps][i % kScanWarps] = kKeyNone;
    S.wrow[i / kScanWarps][i % kScanWarps] = kRowNone;
  }
  if (tid < nq) {
    S.sany[tid] = 0;
    // Running best of the whole grid (pruning bound); stale values are fine.
    const uint64_t g0 = *reinterpret_cast<volatile unsigned long long *>(a.gbest + G.q_begin + tid);
#pragma unroll
    for (int w = 0; w < kScanWarps; ++w) S.gb[tid][w] = g0;
  }
  __syncthreads();
}

// Summary of a run of consecutive rows: which flag bits and accelerator keys
// (id mod 64) occur, and the cheapest price per price column. Static per
// catalog, so it is computed once at ingest for every 128-row chunk (the
// "zone map"); the streaming kernel derives it from the rows it holds.
struct RowSummary {
  uint32_t fl_or, sg_lo, sg_hi;
  uint32_t grp;       // bit (group % 32) of every fixed-host group present
  uint64_t wmin[2];   // price keys (kKeyNone = no priced valid row)
};
static_assert(sizeof(RowSummary) == 32, "zone map entry layout");

// Queries of the staged chunk that can match anything in rows with summary
// `z`: lane q tests query q -- required flag bits present, a wanted
// accelerator key present, and the cheapest price not already beaten by the
// grid-wide running best (branch-and-bound on the argmin; table queries need
// every matching row and are never bounded). One ballot for <= 32 queries.
__device__ __forceinline__ uint32_t active_queries(const ScanShared &S, int nq,
                                                   const RowSummary &z) {
  const int lane = threadIdx.x & 31;
  bool pass = false;
  if (lane < nq) {
    const QueryS &L = S.q[lane].s;
    const uint32_t rq = L.req_flags;
    pass = ((z.fl_or & rq) == rq) && ((z.grp & L.grp_bit) == L.grp_bit) &&
           (!(L.qflags & SKYOPT_Q_ACC) ||
            (((L.sig_lo & z.sg_lo) | (L.sig_hi & z.sg_hi)) != 0u));
    const bool prunable = !(L.qflags & (SKYOPT_Q_LIST | SKYOPT_Q_FUZZY));
    if (prunable && z.wmin[L.price_col ? 1 : 0] > S.gb[lane][threadIdx.x >> 5]) pass = false;
  }
  return __ballot_sync(0xFFFFFFFFu, pass);
}

// Summary of this warp's rows from the registers (streaming kernel).
template <int RPT>
__device__ __forceinline__ RowSummary summarize_rows(
    const ScanGroup &G, int64_t base, const double (&od)[RPT], const double (&sp)[RPT],
    const uint32_t (&ak)[RPT], const uint32_t (&fl)[RPT]) {
  RowSummary z;
  uint32_t fl_or = 0, sg_lo = 0, sg_hi = 0, grp = 0;
  uint64_t k[2] = {kKeyNone, kKeyNone};
#pragma unroll
  for (int j = 0; j < RPT; ++j) {
    const uint32_t f = (base + j < G.row_end) ? fl[j] : 0u;
    fl_or |= f;
    if ((f & SKYOPT_F_VALID) && (f >> 8)) grp |= 1u << ((f >> 8) & 31u);
    if (ak[j] != SKYOPT_NONE16 && (f & SKYOPT_F_VALID)) {
      if (ak[j] & 32u) sg_hi |= 1u << (ak[j] & 31u); else sg_lo |= 1u << (ak[j] & 31u);
    }
    if (f & SKYOPT_F_VALID) {
      if ((G.need & 1u) && od[j] == od[j]) k[0] = min(k[0], price_key(od[j]));
      if ((G.need & 2u) && sp[j] == sp[j]) k[1] = min(k[1], price_key(sp[j]));
    }
  }
  z.fl_or = __reduce_or_sync(0xFFFFFFFFu, fl_or & 0xFFu);
  z.sg_lo = __reduce_or_sync(0xFFFFFFFFu, sg_lo);
  z.sg_hi = __reduce_or_sync(0xFFFFFFFFu, sg_hi);
  z.grp = __reduce_or_sync(0xFFFFFFFFu, grp);
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    const uint32_t h = __reduce_min_sync(0xFFFFFFFFu, (uint32_t)(k[c] >> 32));
    const uint32_t l = __reduce_min_sync(
        0xFFFFFFFFu, ((uint32_t)(k[c] >> 32) == h) ? (uint32_t)k[c] : 0xFFFFFFFFu);
    z.wmin[c] = ((uint64_t)h << 32) | l;
  }
  return z;
}

// Score this thread's RPT rows (already in registers) against the `active`
// staged queries; per-warp running minima accumulate in S.wkey / S.wrow.
// (Variants that turn the fp64 columns into order-preserving integer keys --
// B200 issues only one fp64 warp-instruction per cycle per SM,
// tools/fp64_probe.cu -- were measured 1-3 us slower on cfg4: the inner loop
// is bound by its dependent-issue latency at two to six resident warps per
// scheduler, not by the fp64 pipe, and 64-bit integer compares are two
// instructions each.)
template <int RPT>
__device__ __forceinline__ void score_rows(
    const ScanArgs &a, const ScanGroup &G, ScanShared &S, int64_t base, uint32_t active,
    const double (&od)[RPT], const double (&sp)[RPT], const double (&vc)[RPT],
    const double (&mm)[RPT], const uint32_t (&ak)[RPT], const uint32_t (&rg)[RPT],
    const uint32_t (&zn)[RPT], const uint32_t (&fl)[RPT],
    unsigned long long *trace = nullptr) {
  const CatDev &cat = a.cat;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int trace_n = 0;
  // Per-row integer key, computed once and kept in two registers per row:
  //   klo = flags | region << 16,  khi = zone | accelerator key << 16
  // ("no accelerator" becomes key 32 * SKYOPT_ACC_SET_WORDS, whose bitmask
  // word is the zero word after every set).
  uint32_t klo[RPT], khi[RPT];
#pragma unroll
  for (int j = 0; j < RPT; ++j) {
    const uint32_t f = (base + j < G.row_end) ? fl[j] : 0u;
    const uint32_t key = (ak[j] == SKYOPT_NONE16) ? (uint32_t)(32 * SKYOPT_ACC_SET_WORDS) : ak[j];
    klo[j] = f | (rg[j] << 16);
    khi[j] = zn[j] | (key << 16);
  }
  while (active) {
    const int q = __ffs(active) - 1;
    active &= active - 1;
    const QueryS &Q = S.q[q].s;
    const uint32_t qf = Q.qflags;
    if (trace && lane == 0 && trace_n < 30) {  // profiling (SKYOPT_DEBUG & 4)
      trace[4 * trace_n] = (unsigned long long)S.q[q].qid;
      trace[4 * trace_n + 1] = (unsigned long long)clock64();
    }
    uint32_t m1 = 0, mf = 0;
    {
      const uint32_t mlo = Q.mask_lo, mhi = Q.mask_hi, vlo = Q.val_lo, vhi = Q.val_hi;
#pragma unroll
      for (int j = 0; j < RPT; ++j) {
        const uint32_t t = ((klo[j] ^ vlo) & mlo) | ((khi[j] ^ vhi) & mhi);
        m1 |= (uint32_t)(t == 0u) << j;
      }
    }
    if (qf & SKYOPT_Q_ACC) {
      uint32_t me = 0;
#pragma unroll
      for (int j = 0; j < RPT; ++j)
        me |= ((S.q[q].set[0][khi[j] >> 21] >> ((khi[j] >> 16) & 31u)) & 1u) << j;
      if (qf & SKYOPT_Q_FUZZY) {
#pragma unroll
        for (int j = 0; j < RPT; ++j)
          mf |= ((S.q[q].set[1][khi[j] >> 21] >> ((khi[j] >> 16) & 31u)) & 1u) << j;
        mf &= m1;
      }
      m1 &= me;
    }
    if (Q.disk_op != 0 && (m1 | mf)) {
      // AWS local-disk size test (common.py:499-504); rare, so the column is
      // gathered on demand.
#pragma unroll
      for (int j = 0; j < RPT; ++j) {
        if (((m1 | mf) >> j) & 1u) {
          const double total = cat.disk_total ? __ldg(cat.disk_total + base + j) : 0.0;
          const bool okd = Q.disk_op == SKYOPT_DISK_GE
                               ? (total >= Q.disk_size)
                               : (fabs(total - Q.disk_size) < 1.0);
          if (!okd) { m1 &= ~(1u << j); mf &= ~(1u << j); }
        }
      }
    }
    uint64_t bkey = kKeyNone;
    uint32_t brow = kRowNone;
    if (trace && lane == 0 && trace_n < 30) trace[4 * trace_n + 2] = (unsigned long long)clock64();
    if (m1) {
      S.sany[q] = 1u;  // benign race: every writer stores 1
      // Second stage, branch-free over the thread's RPT rows (the operators
      // are per query, so they select thresholds instead of code paths): the
      // rows' fp64 compares are independent and pipeline.
      const uint32_t f2 = Q.flags2;
      const int mop = Q.mem_op, pcol = Q.price_col;
      const bool nocpu = Q.cpus_op == 0, nomem = mop == 0, ratio = mop == SKYOPT_OP_RATIO;
      const double clo = Q.cpu_lo, chi = Q.cpu_hi, mlo = Q.mem_lo, mhi = Q.mem_hi;
      const double cap = Q.cap;
      uint32_t okm = 0;
#pragma unroll
      for (int j = 0; j < RPT; ++j) {
        // 'rx': MemoryGiB >= vCPUs * r (common.py:476), else the interval
        const double lo = ratio ? __dmul_rn(vc[j], mlo) : mlo;
        const bool okc = nocpu | ((vc[j] >= clo) & (vc[j] <= chi));
        const bool okr = nomem | ((mm[j] >= lo) & (mm[j] <= mhi));
        const bool okj = ((m1 >> j) & 1u) & ((klo[j] & f2) == f2) & okc & okr;
        okm |= (uint32_t)okj << j;
        const double p = pcol ? sp[j] : od[j];
        const uint64_t key = (okj & (p <= cap)) ? price_key(p) : kKeyNone;  // NaN: false
        if (key < bkey) { bkey = key; brow = (uint32_t)(base + j); }
      }
      if ((qf & SKYOPT_Q_LIST) && okm) {
        // per-instance-type minima for the sorted list (catalog API only)
#pragma unroll
        for (int j = 0; j < RPT; ++j) {
          if (!((okm >> j) & 1u)) continue;
          const double p = pcol ? sp[j] : od[j];
          uint64_t key = kKeyNone;
          if (p <= cap) key = price_key(p);
          else if ((qf & SKYOPT_Q_KEEP_NAN) && p != p) key = kKeyNaN;
          if (key == kKeyNone) continue;
          const int inst = __ldg(cat.inst_id + base + j);
          if (inst >= 0) {
            const int local = inst - __ldg(&cat.cloud_inst_offsets[Q.cloud]);
            atomicMin(&a.list_min[S.q[q].list_base + local], (unsigned long long)key);
          }
        }
      }
      // cannot beat (or tie) what the grid already has: no reduction needed
      if (bkey > S.gb[q][threadIdx.x >> 5]) brow = kRowNone;
    }
    if (mf) {
      // Fuzzy table: min 'Price' per accelerator key (common.py:661-667).
#pragma unroll
      for (int j = 0; j < RPT; ++j) {
        if (!((mf >> j) & 1u)) continue;
        const double p = (G.need & 1u) ? od[j] : __ldg(cat.price + base + j);
        const uint64_t key = (p == p) ? price_key(p) : kKeyNaN;
        atomicMin(&a.fuzzy_min[S.q[q].fuzzy_base + (khi[j] >> 16)],
                  (unsigned long long)key);
      }
    }
    if (trace && lane == 0 && trace_n < 30) { trace[4 * trace_n + 3] = (unsigned long long)clock64(); ++trace_n; }
    // Warp argmin of (price key, row) with three REDUX steps; skipped when no
    // lane has a candidate (the common case for selective queries). Lane 0
    // folds the result into the warp's running minimum.
    if (__any_sync(0xFFFFFFFFu, brow != kRowNone)) {
      const uint32_t khi32 = (uint32_t)(bkey >> 32);
      const uint32_t mhi32 = __reduce_min_sync(0xFFFFFFFFu, khi32);
      uint32_t mlo32, mr;
      const uint32_t tied = __ballot_sync(0xFFFFFFFFu, khi32 == mhi32);
      if ((tied & (tied - 1)) == 0) {
        // one lane holds the minimum of the high word (prices are almost
        // always distinct there): broadcast its key and row
        const int src = __ffs(tied) - 1;
        mlo32 = __shfl_sync(0xFFFFFFFFu, (uint32_t)bkey, src);
        mr = __shfl_sync(0xFFFFFFFFu, brow, src);
      } else {
        const uint32_t klo32 = (khi32 == mhi32) ? (uint32_t)bkey : 0xFFFFFFFFu;
        mlo32 = __reduce_min_sync(0xFFFFFFFFu, klo32);
        const uint32_t kr = (khi32 == mhi32 && klo32 == mlo32) ? brow : kRowNone;
        mr = __reduce_min_sync(0xFFFFFFFFu, kr);
      }
      __syncwarp();  // every lane has read the warp's bound for this query
      if (lane == 0) {
        const uint64_t k = ((uint64_t)mhi32 << 32) | mlo32;
        const uint64_t ok_ = S.wkey[q][warp];
        if (k < ok_ || (k == ok_ && mr < S.wrow[q][warp])) {
          S.wkey[q][warp] = k;
          S.wrow[q][warp] = mr;
        }
        if (k < S.gb[q][warp]) {
          // tighten this warp's bound and the grid's (any achieved key is
          // a valid bound)
          S.gb[q][warp] = k;
          atomicMin(a.gbest + G.q_begin + q, (unsigned long long)k);
        }
      }
      __syncwarp();  // ... and sees the tightened one from here on
    }
  }
}

// Block reduction of the per-warp minima -> one partial per (query, block).
__device__ __forceinline__ void finish_block(const ScanArgs &a, const ScanGroup &G,
                                             ScanShared &S, int block_in_group) {
  __syncthreads();
  const int tid = threadIdx.x;
  if (tid < G.q_count) {
    uint64_t k = kKeyNone;
    uint32_t r = kRowNone;
#pragma unroll
    for (int w = 0; w < kScanWarps; ++w) {
      const uint64_t kw = S.wkey[tid][w];
      const uint32_t rw = S.wrow[tid][w];
      if (kw < k || (kw == k && rw < r)) { k = kw; r = rw; }
    }
    ScanPartial out;
    out.key = k; out.row = r; out.pad_ = S.sany[tid];
    a.partials[(int64_t)S.q[tid].partial_base + block_in_group] = out;
  }
}

// K1, small catalogs: one tile of 256*RPT rows per block, rows go straight
// from global memory to registers.
constexpr int kZoneRows = 128;  // rows per zone-map entry

template <int RPT>
__global__ void __launch_bounds__(kScanThreads, kScanBlocksPerSM) scan_kernel(ScanArgs a) {
  __shared__ __align__(16) ScanShared S;
  const int vb = permuted_block(a);
  const ScanGroup G = find_group(a, vb);
  const int slot = vb - G.block0;  // partial slot of this block within its group
  // the group's tiles: a run of consecutive tiles, or an explicit list
  const int tile = (G.list0 < 0) ? G.tile0 + slot : __ldg(a.tile_list + G.list0 + slot);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nq = G.q_count;
  if (blockIdx.x == 0 && tid == 0 && a.zero_flag) *a.zero_flag = 0;
  mark(a, 0);
  const int64_t base =
      (int64_t)G.row_begin + (int64_t)tile * (kScanThreads * RPT) + tid * RPT;
  const int64_t warp_row = base - (int64_t)lane * RPT;

  // ---- phase A: zone-map test, lane q <-> query q, operands straight from
  // global memory (the warp's 32-byte summary of its rows, the query's
  // 32-byte test record, the grid-wide running best). Cloud ranges are
  // 128-row aligned, so a summary never mixes clouds; with RPT < 4 several
  // warps share one, which is merely less tight. (Letting one warp test all
  // eight chunks of the tile saves a quarter of the kernel's instructions and
  // was measured slower: the block is latency-bound, not issue-bound.)
  bool pass = false;
  QueryTest qt;
  unsigned long long gb = kKeyNone;
  if (lane < nq) {
    const uint4 *tp = reinterpret_cast<const uint4 *>(a.qtests + G.q_begin + lane);
    const uint4 t0 = __ldg(tp), t1 = __ldg(tp + 1);
    qt.req_flags = t0.x; qt.grp_bit = t0.y; qt.sig_lo = t0.z; qt.sig_hi = t0.w;
    qt.qflags = t1.x; qt.price_col = t1.y; qt.partial_base = (int32_t)t1.z;
    // stale values of the running best are fine: any achieved key is a bound
    gb = *reinterpret_cast<volatile unsigned long long *>(a.gbest + G.q_begin + lane);
  }
  if (warp_row < G.row_end) {
    const uint4 *zp = reinterpret_cast<const uint4 *>(a.cat.zone_map + warp_row / kZoneRows);
    const uint4 z0 = __ldg(zp), z1 = __ldg(zp + 1);
    if (lane < nq) {
      pass = ((z0.x & qt.req_flags) == qt.req_flags) && ((z0.w & qt.grp_bit) == qt.grp_bit) &&
             (!(qt.qflags & SKYOPT_Q_ACC) || (((qt.sig_lo & z0.y) | (qt.sig_hi & z0.z)) != 0u));
      // branch-and-bound on the argmin: nothing in these rows is cheaper than
      // what the grid already has (table queries need every matching row)
      const uint64_t wmin = qt.price_col ? (((uint64_t)z1.w << 32) | z1.z)
                                         : (((uint64_t)z1.y << 32) | z1.x);
      if (!(qt.qflags & (SKYOPT_Q_LIST | SKYOPT_Q_FUZZY)) && wmin > gb) pass = false;
    }
  }
  const uint32_t active = __ballot_sync(0xFFFFFFFFu, pass);
  if (lane == 0) S.wact[warp] = active;
  __syncthreads();
  uint32_t wanted = 0;  // queries some warp of the block has to score
#pragma unroll
  for (int w = 0; w < kScanWarps; ++w) wanted |= S.wact[w];
  if (wanted == 0) {
    // The summaries prove that no row of this tile can match or improve any
    // query: one empty partial per query and the block is done, without ever
    // staging the constraint vectors.
    if (tid < nq) {
      ScanPartial out;
      out.key = kKeyNone; out.row = kRowNone; out.pad_ = 0;
      a.partials[(int64_t)qt.partial_base + slot] = out;
    }
    mark(a, 3);
    return;
  }

  // ---- phase B: stage the surviving queries' records (16-byte loads, one
  // record per warp at a time), initialise the per-warp minima.
  {
    const uint4 *src = reinterpret_cast<const uint4 *>(a.squeries + G.q_begin);
    uint4 *dst = reinterpret_cast<uint4 *>(S.q);
    constexpr int kWords = (int)(sizeof(ScanQuery) / 16);
    static_assert(kWords <= 32, "one lane per 16-byte word of a record");
    uint32_t todo = wanted;
    for (int k = 0; todo; ++k) {
      const int q = __ffs(todo) - 1;
      todo &= todo - 1;
      if ((k & (kScanWarps - 1)) == warp && lane < kWords)
        dst[q * kWords + lane] = __ldg(src + q * kWords + lane);
    }
    for (int i = tid; i < nq * kScanWarps; i += kScanThreads) {
      S.wkey[i / kScanWarps][i % kScanWarps] = kKeyNone;
      S.wrow[i / kScanWarps][i % kScanWarps] = kRowNone;
    }
    if (tid < nq) {
      S.sany[tid] = 0;
#pragma unroll
      for (int w = 0; w < kScanWarps; ++w) S.gb[tid][w] = gb;
    }
  }
  __syncthreads();
  mark(a, 1);
  // ---- phase C: only warps with something to score stream their rows
  // (32 B per row); the others are proven non-matching / non-improving by the
  // summary. (Measured and rejected: several tiles per block -- the per-tile
  // latencies serialise inside the block, while independent blocks overlap
  // them; dealing the surviving (chunk, query) pairs evenly to the block's
  // warps -- no gain, more registers.)
  if (active) {
    double od[RPT], sp[RPT], vc[RPT], mm[RPT];
    uint32_t ak[RPT], rg[RPT], zn[RPT], fl[RPT];
    if (G.need & 1u) load_f64<RPT>(a.cat.price, base, od);
    if (G.need & 2u) load_f64<RPT>(a.cat.spot, base, sp);
    load_f64<RPT>(a.cat.vcpus, base, vc);
    load_f64<RPT>(a.cat.mem, base, mm);
    load_u16<RPT>(a.cat.acc_key, base, ak);
    load_u16<RPT>(a.cat.region_id, base, rg);
    load_u16<RPT>(a.cat.zone_id, base, zn);
    load_u16<RPT>(a.cat.flags, base, fl);
    unsigned long long *trace = nullptr;
    if ((a.debug & 4u) && vb == (int)a.trace_vb && warp == (int)a.trace_warp)
      trace = a.timeline + (size_t)a.n_blocks * 8;
    score_rows<RPT>(a, G, S, base, active, od, sp, vc, mm, ak, rg, zn, fl, trace);
    if (trace && lane == 0) { trace[126] = (unsigned long long)clock64(); trace[127] = __popc(active); }
  }
  mark(a, 2);
  // Block reduction of the per-warp minima -> one partial per (query, block).
  __syncthreads();
  if (tid < nq) {
    uint64_t k = kKeyNone;
    uint32_t r = kRowNone;
    uint32_t any = 0;
    if ((wanted >> tid) & 1u) {
#pragma unroll
      for (int w = 0; w < kScanWarps; ++w) {
        const uint64_t kw = S.wkey[tid][w];
        const uint32_t rw = S.wrow[tid][w];
        if (kw < k || (kw == k && rw < r)) { k = kw; r = rw; }
      }
      any = S.sany[tid];
    }
    ScanPartial out;
    out.key = k; out.row = r; out.pad_ = any;
    a.partials[(int64_t)qt.partial_base + slot] = out;
  }
  mark(a, 3);
}

// ---- TMA (cp.async.bulk) + mbarrier plumbing for the streaming kernel ------
// K1, queue form: a block owns `tiles_per_block` tiles of its group (strided
// over the group's tile list, so neighbouring -- similarly expensive -- tiles
// land in different blocks). The zone-map entries of all its 128-row chunks
// are fetched while the query records are being staged; each warp then tests
// its share of the chunks (lane q <-> query q, one ballot per chunk) and pushes
// the survivors as work entries -- a chunk and at most two of its surviving
// queries -- into a shared-memory queue. All warps pop entries until the queue
// is empty: scoring one (chunk, query) pair is a ~2000-cycle dependent chain,
// so the block's throughput comes from every resident warp working on a
// different pair, whichever chunk it came from.
constexpr int kQueueChunks = kScanThreads;  // one fetched zone-map entry per thread
constexpr int kQueueEntries = 1024;
struct QueueShared {
  uint4 z0[kQueueChunks], z1[kQueueChunks];  // zone-map entries
  int32_t row[kQueueChunks];                 // first row of the chunk, -1 = none
  uint32_t cmask[kQueueChunks];              // surviving queries per chunk
  uint32_t emask[kQueueEntries];             // entry: queries to score ...
  uint16_t echunk[kQueueEntries];            // ... on this chunk
  int n_pairs, n_entries, next;
};

__global__ void __launch_bounds__(kScanThreads, kScanBlocksPerSM) scan_queue_kernel(ScanArgs a) {
  constexpr int RPT = 4;
  constexpr int kTileRows = kScanThreads * RPT;
  constexpr int kChunksPerTile = kTileRows / kZoneRows;
  __shared__ __align__(16) ScanShared S;
  __shared__ __align__(16) QueueShared Q;
  const int vb = permuted_block(a);
  const ScanGroup G = find_group(a, vb);
  const int slot = vb - G.block0;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nq = G.q_count;
  if (blockIdx.x == 0 && tid == 0 && a.zero_flag) *a.zero_flag = 0;
  mark(a, 0);
  if (tid == 0) { Q.n_pairs = 0; Q.n_entries = 0; Q.next = 0; }

  // this thread fetches the entry of chunk c of tile (slot + k * blocks)
  {
    const int k = tid / kChunksPerTile, c = tid % kChunksPerTile;
    const int tidx = slot + k * G.n_tiles;
    int64_t crow = -1;
    uint4 z0 = make_uint4(0, 0, 0, 0), z1 = make_uint4(0, 0, 0, 0);
    if (k < G.tiles_per_block && tidx < G.total_tiles) {
      const int tile = (G.list0 < 0) ? G.tile0 + tidx : __ldg(a.tile_list + G.list0 + tidx);
      const int64_t r = (int64_t)G.row_begin + (int64_t)tile * kTileRows + c * kZoneRows;
      if (r < G.row_end) {
        crow = r;
        const uint4 *zp = reinterpret_cast<const uint4 *>(a.cat.zone_map + r / kZoneRows);
        z0 = __ldg(zp); z1 = __ldg(zp + 1);
      }
    }
    Q.z0[tid] = z0; Q.z1[tid] = z1; Q.row[tid] = (int32_t)crow;
  }
  stage_queries(a, G, S);  // all records of the group; ends with a barrier
  mark(a, 1);

  // zone-map test: warp w takes chunks w, w + 8, ...
  const int n_chunks = min(kQueueChunks, G.tiles_per_block * kChunksPerTile);
  {
    uint32_t req = 0, grp = 0, sg_lo = 0, sg_hi = 0, qf = 0, col = 0;
    uint64_t gb = 0;
    if (lane < nq) {
      const QueryS &L = S.q[lane].s;
      req = L.req_flags; grp = L.grp_bit; sg_lo = L.sig_lo; sg_hi = L.sig_hi;
      qf = L.qflags; col = L.price_col ? 1u : 0u; gb = S.gb[lane][threadIdx.x >> 5];
    }
    const bool bounded = !(qf & (SKYOPT_Q_LIST | SKYOPT_Q_FUZZY));
    int pairs = 0;
    for (int ch = warp; ch < n_chunks; ch += kScanWarps) {
      uint32_t m = 0;
      if (Q.row[ch] >= 0) {
        const uint4 z0 = Q.z0[ch], z1 = Q.z1[ch];
        const uint64_t wmin = col ? (((uint64_t)z1.w << 32) | z1.z) : (((uint64_t)z1.y << 32) | z1.x);
        const bool pass = lane < nq && ((z0.x & req) == req) && ((z0.w & grp) == grp) &&
                          (!(qf & SKYOPT_Q_ACC) || (((sg_lo & z0.y) | (sg_hi & z0.z)) != 0u)) &&
                          !(bounded && wmin > gb);
        m = __ballot_sync(0xFFFFFFFFu, pass);
      }
      if (lane == 0) Q.cmask[ch] = m;
      pairs += __popc(m);
    }
    if (lane == 0 && pairs) atomicAdd(&Q.n_pairs, pairs);
  }
  __syncthreads();
  // entries: two queries each while they fit the queue, else whole chunks
  {
    const int split = (Q.n_pairs <= kQueueEntries) ? (int)a.qsplit : 32;
    if (tid < n_chunks) {
      uint32_t m = Q.cmask[tid];
      while (m) {
        uint32_t e = 0;
        for (int n = 0; n < split && m; ++n) { const uint32_t low = m & (0u - m); e |= low; m ^= low; }
        const int i = atomicAdd(&Q.n_entries, 1);
        Q.emask[i] = e; Q.echunk[i] = (uint16_t)tid;
      }
    }
  }
  __syncthreads();
  if ((a.debug & 2u) && tid == 0) {  // profiling: work of the block
    a.timeline[(size_t)blockIdx.x * 8 + 4] =
        (unsigned long long)Q.n_entries | ((unsigned long long)Q.n_pairs << 32);
    a.timeline[(size_t)blockIdx.x * 8 + 5] = (unsigned long long)G.block0 | ((unsigned long long)nq << 32);
    a.timeline[(size_t)blockIdx.x * 8 + 6] = global_ns();
  }
  const int n_entries = Q.n_entries;
  for (;;) {
    int i = 0;
    if (lane == 0) i = atomicAdd(&Q.next, 1);
    i = __shfl_sync(0xFFFFFFFFu, i, 0);
    if (i >= n_entries) break;
    const int ch = Q.echunk[i];
    const int64_t base = (int64_t)Q.row[ch] + lane * RPT;
    uint32_t active = Q.emask[i];
    // the bound may have tightened since the chunk was tested
    {
      bool drop = false;
      if (lane < nq && ((active >> lane) & 1u)) {
        const QueryS &L = S.q[lane].s;
        const uint4 z1 = Q.z1[ch];
        const uint64_t wmin = L.price_col ? (((uint64_t)z1.w << 32) | z1.z) : (((uint64_t)z1.y << 32) | z1.x);
        drop = !(L.qflags & (SKYOPT_Q_LIST | SKYOPT_Q_FUZZY)) && wmin > S.gb[lane][threadIdx.x >> 5];
      }
      active &= ~__ballot_sync(0xFFFFFFFFu, drop);
    }
    if (!active) continue;
    double od[RPT], sp[RPT], vc[RPT], mm[RPT];
    uint32_t ak[RPT], rg[RPT], zn[RPT], fl[RPT];
    if (G.need & 1u) load_f64<RPT>(a.cat.price, base, od);
    if (G.need & 2u) load_f64<RPT>(a.cat.spot, base, sp);
    load_f64<RPT>(a.cat.vcpus, base, vc);
    load_f64<RPT>(a.cat.mem, base, mm);
    load_u16<RPT>(a.cat.acc_key, base, ak);
    load_u16<RPT>(a.cat.region_id, base, rg);
    load_u16<RPT>(a.cat.zone_id, base, zn);
    load_u16<RPT>(a.cat.flags, base, fl);
    score_rows<RPT>(a, G, S, base, active, od, sp, vc, mm, ak, rg, zn, fl);
  }
  mark(a, 2);
  finish_block(a, G, S, slot);
  mark(a, 3);
}

__device__ __forceinline__ uint32_t smem_u32(const void *p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;"
               ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes,
                                         uint64_t *bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
      ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

constexpr int kStreamRPT = 4;
constexpr int kStreamTile = kScanThreads * kStreamRPT;   // 1024 rows
constexpr int kStreamStages = 2;
// one stage: price, spot, vcpus, mem (f64) + acc_key, region, zone, flags (u16)
constexpr int kStageBytes = kStreamTile * (4 * 8 + 4 * 2);

struct StreamStage {
  double od[kStreamTile], sp[kStreamTile], vc[kStreamTile], mm[kStreamTile];
  uint16_t ak[kStreamTile], rg[kStreamTile], zn[kStreamTile], fl[kStreamTile];
};
static_assert(sizeof(StreamStage) == kStageBytes, "stage layout");

// K1, large catalogs: each block owns `tiles_per_block` consecutive tiles of
// one (cloud, query chunk) group. Thread 0 keeps two tiles in flight with
// cp.async.bulk (TMA) into shared memory, completion is signalled through
// mbarriers; all threads copy their rows out to registers, hand the stage
// back and score the rows while the next tiles stream in. The constraint
// vectors are staged once per block.
__global__ void __launch_bounds__(kScanThreads, 512 / kScanThreads) scan_stream_kernel(ScanArgs a) {
  extern __shared__ __align__(128) unsigned char stream_smem[];
  StreamStage *stages = reinterpret_cast<StreamStage *>(stream_smem);
  __shared__ __align__(16) ScanShared S;
  __shared__ __align__(8) uint64_t full[kStreamStages];
  const int vb = permuted_block(a);
  const ScanGroup G = find_group(a, vb);
  const int blk = vb - G.block0;
  const int tid = threadIdx.x;
  if (blockIdx.x == 0 && tid == 0 && a.zero_flag) *a.zero_flag = 0;
  // Block `blk` of the group owns tiles blk, blk + n_blocks, blk + 2*n_blocks,
  // ...: every block gets the same mix of cheap and expensive catalog regions.
  const int stride = G.n_tiles;
  const int ntiles = (G.total_tiles - blk + stride - 1) / stride;
  const CatDev &cat = a.cat;

  auto issue = [&](int i) {
    // tile t0 + i -> stage i % kStreamStages (thread 0 only)
    StreamStage &st = stages[i % kStreamStages];
    uint64_t *bar = &full[i % kStreamStages];
    const int64_t row = (int64_t)G.row_begin + (int64_t)(blk + i * stride) * kStreamTile;
    uint32_t bytes = kStreamTile * (2 * 8 + 4 * 2);
    if (G.need & 1u) bytes += kStreamTile * 8;
    if (G.need & 2u) bytes += kStreamTile * 8;
    mbar_expect_tx(bar, bytes);
    if (G.need & 1u) bulk_g2s(st.od, cat.price + row, kStreamTile * 8, bar);
    if (G.need & 2u) bulk_g2s(st.sp, cat.spot + row, kStreamTile * 8, bar);
    bulk_g2s(st.vc, cat.vcpus + row, kStreamTile * 8, bar);
    bulk_g2s(st.mm, cat.mem + row, kStreamTile * 8, bar);
    bulk_g2s(st.ak, cat.acc_key + row, kStreamTile * 2, bar);
    bulk_g2s(st.rg, cat.region_id + row, kStreamTile * 2, bar);
    bulk_g2s(st.zn, cat.zone_id + row, kStreamTile * 2, bar);
    bulk_g2s(st.fl, cat.flags + row, kStreamTile * 2, bar);
  };

  if (tid == 0) {
    for (int s = 0; s < kStreamStages; ++s) mbar_init(&full[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (tid == 0)
    for (int i = 0; i < min(kStreamStages, ntiles); ++i) issue(i);
  stage_queries(a, G, S);

  for (int i = 0; i < ntiles; ++i) {
    const int s = i % kStreamStages;
    mbar_wait(&full[s], (uint32_t)((i / kStreamStages) & 1));
    const StreamStage &st = stages[s];
    double od[kStreamRPT], sp[kStreamRPT], vc[kStreamRPT], mm[kStreamRPT];
    uint32_t ak[kStreamRPT], rg[kStreamRPT], zn[kStreamRPT], fl[kStreamRPT];
    const int r0 = tid * kStreamRPT;
    auto ld4 = [&](const double *col, double (&out)[kStreamRPT]) {
      const double2 x = *reinterpret_cast<const double2 *>(col + r0);
      const double2 y = *reinterpret_cast<const double2 *>(col + r0 + 2);
      out[0] = x.x; out[1] = x.y; out[2] = y.x; out[3] = y.y;
    };
    auto ld4u = [&](const uint16_t *col, uint32_t (&out)[kStreamRPT]) {
      const uint2 x = *reinterpret_cast<const uint2 *>(col + r0);
      out[0] = x.x & 0xFFFF; out[1] = x.x >> 16; out[2] = x.y & 0xFFFF; out[3] = x.y >> 16;
    };
    if (G.need & 1u) ld4(st.od, od);
    if (G.need & 2u) ld4(st.sp, sp);
    ld4(st.vc, vc); ld4(st.mm, mm);
    ld4u(st.ak, ak); ld4u(st.rg, rg); ld4u(st.zn, zn); ld4u(st.fl, fl);
    __syncthreads();  // every thread has its rows: the stage can be refilled
    if (tid == 0 && i + kStreamStages < ntiles) issue(i + kStreamStages);
    const int64_t base =
        (int64_t)G.row_begin + (int64_t)(blk + i * stride) * kStreamTile + r0;
    const RowSummary z = summarize_rows<kStreamRPT>(G, base, od, sp, ak, fl);
    const uint32_t active = active_queries(S, G.q_count, z);
    if (active)
      score_rows<kStreamRPT>(a, G, S, base, active, od, sp, vc, mm, ak, rg, zn, fl);
  }
  finish_block(a, G, S, blk);
}

// One warp per query: reduce the per-tile partials.
__global__ void finalize_kernel(CatDev cat, int n_queries,
                                const int32_t *__restrict__ partial_base,
                                const int32_t *__restrict__ partial_count,
                                const ScanPartial *__restrict__ partials,
                                ScanFinal *__restrict__ finals,
                                uint32_t *__restrict__ any1,
                                int32_t *__restrict__ err_flag) {
  const int q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (blockIdx.x == 0 && threadIdx.x == 0) *err_flag = 0;
  if (q >= n_queries) return;
  const int64_t pb = partial_base[q];
  const int n = partial_count[q];
  uint64_t k = kKeyNone;
  uint32_t r = kRowNone;
  uint32_t any = 0;
  for (int i = lane; i < n; i += 32) {
    const ScanPartial p = partials[pb + i];
    any |= p.pad_;
    if (p.key < k || (p.key == k && p.row < r)) { k = p.key; r = p.row; }
  }
  any = __reduce_or_sync(0xFFFFFFFFu, any);
  for (int off = 16; off; off >>= 1) {
    const uint64_t ok = __shfl_xor_sync(0xFFFFFFFFu, k, off);
    const uint32_t orow = __shfl_xor_sync(0xFFFFFFFFu, r, off);
    if (ok < k || (ok == k && orow < r)) { k = ok; r = orow; }
  }
  if (lane == 0) {
    ScanFinal f;
    f.key = k;
    f.row = (r == kRowNone) ? -1 : (int32_t)r;
    f.inst = (r == kRowNone) ? -1 : cat.inst_id[r];
    finals[q] = f;
    any1[q] = any;
  }
}

// ---------------------------------------------------------------------------
// Block-wide bitonic sort of (k1, k2) pairs in shared memory, n = power of 2.
__device__ __forceinline__ void bitonic_sort2(uint64_t *k1, uint64_t *k2, int n) {
  for (int size = 2; size <= n; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      __syncthreads();
      for (int i = threadIdx.x; i < (n >> 1); i += blockDim.x) {
        const int lo = 2 * i - (i & (stride - 1));
        const int hi = lo + stride;
        const bool up = ((lo & size) == 0);
        const uint64_t a1 = k1[lo], a2 = k2[lo], b1 = k1[hi], b2 = k2[hi];
        const bool gt = (a1 > b1) || (a1 == b1 && a2 > b2);
        if (gt == up) { k1[lo] = b1; k2[lo] = b2; k1[hi] = a1; k2[hi] = a2; }
      }
    }
  }
  __syncthreads();
}

// Sort the first `n` (k1, k2) pairs (keys unique; entries >= n hold the
// "none" key). Small inputs -- the usual case: one instance type's rows -- are
// ranked by counting (each element counts the smaller ones: n broadcast reads,
// no barriers in the loop); larger ones fall back to the bitonic network.
constexpr int kCountSortMax = 256;
__device__ __forceinline__ void sort_pairs(uint64_t *k1, uint64_t *k2, uint64_t *t1,
                                           uint64_t *t2, int n, int sort_n) {
  if (n > kCountSortMax) { bitonic_sort2(k1, k2, sort_n); return; }
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const uint64_t a1 = k1[i], a2 = k2[i];
    int rank = 0;
    for (int j = 0; j < n; ++j) {
      const uint64_t b1 = k1[j], b2 = k2[j];
      rank += (b1 < a1) || (b1 == a1 && b2 < a2);
    }
    t1[rank] = a1; t2[rank] = a2;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) { k1[i] = t1[i]; k2[i] = t2[i]; }
  __syncthreads();
}

// Sorted tables of skyopt_scan: block per (query, kind). kind 0 = instance
// types by min price (common.py:692-693), kind 1 = fuzzy accelerator keys by
// min Price (common.py:665-667).
__global__ void list_kernel(CatDev cat, const SkyoptQuery *__restrict__ queries,
                            int kind, const int64_t *__restrict__ base,
                            const unsigned long long *__restrict__ table,
                            int cap, int sort_n, int32_t *__restrict__ out_ids,
                            double *__restrict__ out_prices,
                            int32_t *__restrict__ out_count) {
  extern __shared__ uint64_t smem_u64[];
  uint64_t *k1 = smem_u64, *k2 = smem_u64 + sort_n;
  __shared__ int s_n;
  const int q = blockIdx.x;
  const SkyoptQuery Q = queries[q];
  const uint32_t want = kind == 0 ? SKYOPT_Q_LIST : SKYOPT_Q_FUZZY;
  if (!(Q.qflags & want)) {
    if (threadIdx.x == 0) out_count[q] = 0;
    return;
  }
  const int n_entries = kind == 0 ? cat.cloud_inst_offsets[Q.cloud + 1] -
                                        cat.cloud_inst_offsets[Q.cloud]
                                  : cat.n_acc_keys;
  const int id0 = kind == 0 ? cat.cloud_inst_offsets[Q.cloud] : 0;
  if (threadIdx.x == 0) s_n = 0;
  for (int i = threadIdx.x; i < sort_n; i += blockDim.x) { k1[i] = kKeyNone; k2[i] = kKeyNone; }
  __syncthreads();
  const unsigned long long *t = table + base[q];
  for (int i = threadIdx.x; i < n_entries; i += blockDim.x) {
    const uint64_t k = t[i];
    if (k != kKeyNone) {
      const int pos = atomicAdd(&s_n, 1);
      if (pos < sort_n) { k1[pos] = k; k2[pos] = (uint64_t)(id0 + i); }
    }
  }
  __syncthreads();
  const int n = min(s_n, sort_n);
  bitonic_sort2(k1, k2, sort_n);
  const int n_out = min(n, cap);
  for (int i = threadIdx.x; i < n_out; i += blockDim.x) {
    out_ids[(int64_t)q * cap + i] = (int32_t)k2[i];
    out_prices[(int64_t)q * cap + i] =
        k1[i] == kKeyNaN ? __longlong_as_double(0x7FF8000000000000ll) : key_price(k1[i]);
  }
  if (threadIdx.x == 0) out_count[q] = n_out;
}

// ---------------------------------------------------------------------------
// K2: one block per slot.
struct ExpandOut {
  int32_t *slot_count;     // [n_slots]
  int32_t *slot_inst;      // [n_slots]
  int32_t *cand_region;    // candidate buffers at slot_off[s]
  int32_t *cand_zone;
  double *cand_price_a;    // instance price
  double *cand_price_b;    // GCP accelerator price (0 otherwise)
};

// Block-wide reduction of one query's per-block scan partials: the cheapest
// fully-matching row (lowest row id on a price tie) and the any-match bit.
// Every thread gets the result. `red` is scratch for blockDim/32 entries.
struct PartialBest { uint64_t key; uint32_t row; uint32_t any; };
__device__ __forceinline__ PartialBest reduce_partials(
    const ScanPartial *__restrict__ partials, int64_t pb, int n, PartialBest *red) {
  uint64_t k = kKeyNone; uint32_t r = kRowNone, any = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const ScanPartial p = partials[pb + i];
    any |= p.pad_;
    if (p.key < k || (p.key == k && p.row < r)) { k = p.key; r = p.row; }
  }
  for (int off = 16; off; off >>= 1) {
    const uint64_t ok = __shfl_xor_sync(0xFFFFFFFFu, k, off);
    const uint32_t orow = __shfl_xor_sync(0xFFFFFFFFu, r, off);
    if (ok < k || (ok == k && orow < r)) { k = ok; r = orow; }
  }
  any = __reduce_or_sync(0xFFFFFFFFu, any);
  const int warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  __syncthreads();  // `red` may still be read from a previous call
  if ((threadIdx.x & 31) == 0) { red[warp].key = k; red[warp].row = r; red[warp].any = any; }
  __syncthreads();
  PartialBest b = red[0];
  for (int w = 1; w < nw; ++w) {
    const PartialBest o = red[w];
    b.any |= o.any;
    if (o.key < b.key || (o.key == b.key && o.row < b.row)) { b.key = o.key; b.row = o.row; }
  }
  return b;
}

__global__ void expand_kernel(CatDev cat, const SkyoptSlot *__restrict__ slots,
                              const int32_t *__restrict__ partial_base,
                              const int32_t *__restrict__ partial_count,
                              const ScanPartial *__restrict__ partials,
                              const uint32_t *__restrict__ acc_sets,
                              const int64_t *__restrict__ slot_off, int sort_n,
                              int max_regions, int max_zones, ExpandOut out,
                              int32_t *__restrict__ err_flag) {
  extern __shared__ uint64_t smem_u64[];
  uint64_t *k1 = smem_u64;                 // [sort_n] price key
  uint64_t *k2 = k1 + sort_n;              // [sort_n] region|zone|local
  double *bprice = reinterpret_cast<double *>(k2 + sort_n);  // [max_zones]
  int32_t *first_pos = reinterpret_cast<int32_t *>(bprice + max_zones);  // [max_regions]
  __shared__ int s_n;
  __shared__ uint64_t s_t1[kCountSortMax], s_t2[kCountSortMax];  // counting-sort scratch

  const int s = blockIdx.x;
  const SkyoptSlot S = slots[s];
  const int tid = threadIdx.x;
  const int cloud = S.cloud;
  const int reg0 = cat.cloud_region_offsets[cloud];
  const bool has_zones = cat.cloud_n_zones[cloud] > 0;

  // The scan leaves one partial per (query, block); this slot's block folds
  // the partials of the queries it depends on itself (no separate pass).
  __shared__ PartialBest s_red[8];
  int inst = S.inst_id;
  bool empty = false;
  if (S.gate_query >= 0) {
    const PartialBest g = reduce_partials(partials, partial_base[S.gate_query],
                                          partial_count[S.gate_query], s_red);
    if (g.any == 0) empty = true;
  }
  if (S.query >= 0) {
    const PartialBest f = reduce_partials(partials, partial_base[S.query],
                                          partial_count[S.query], s_red);
    if (f.row == kRowNone) empty = true;
    else {
      inst = cat.inst_id[f.row];
      if (inst < 0) empty = true;
    }
  }
  if (empty || (inst < 0 && inst != -2)) {
    if (tid == 0) { out.slot_count[s] = 0; out.slot_inst[s] = -1; }
    return;
  }
  if (tid == 0) s_n = 0;
  for (int i = tid; i < sort_n; i += blockDim.x) { k1[i] = kKeyNone; k2[i] = kKeyNone; }
  for (int i = tid; i < max_regions; i += blockDim.x) first_pos[i] = 0x7FFFFFFF;
  const double kNaN = __longlong_as_double(0x7FF8000000000000ll);
  for (int i = tid; i < max_zones; i += blockDim.x) bprice[i] = kNaN;
  __syncthreads();

  const double *pcol = S.price_col ? cat.spot : cat.price;
  const bool gcp_acc = S.acc_set >= 0;

  // Group A: the rows that define the region/zone order -- the instance
  // type's rows, or (GCP) the accelerator's rows.
  auto push_row = [&](int row) {
    const double p = pcol[row];
    const int rg = cat.region_id[row];
    const int zn = cat.zone_id[row];
    // dropna over [price, Region, AvailabilityZone] (common.py:797-802)
    if (p != p) return;
    if (has_zones && zn == SKYOPT_NONE16) return;
    const int pos = atomicAdd(&s_n, 1);
    if (pos < sort_n) {
      k1[pos] = price_key(p);
      k2[pos] = ((uint64_t)rg << 48) | ((uint64_t)(has_zones ? zn : 0) << 32) |
                (uint32_t)row;
    }
  };
  if (gcp_acc) {
    const uint32_t *set = acc_sets + (int64_t)S.acc_set * SKYOPT_ACC_SET_WORDS;
    for (int k = 0; k < cat.n_acc_keys; ++k) {
      if (!test_bit(set, k)) continue;  // uniform branch
      const int b = cat.acc_row_offsets[k], e = cat.acc_row_offsets[k + 1];
      const int r0 = cat.cloud_row_offsets[cloud], r1 = cat.cloud_row_offsets[cloud + 1];
      for (int i = b + tid; i < e; i += blockDim.x) {
        const int row = cat.acc_rows[i];
        if (row >= r0 && row < r1) push_row(row);
      }
    }
    // Group B: host VM zones with a price (gcp.py:296-322).
    if (inst >= 0) {
      const int b = cat.inst_row_offsets[inst], e = cat.inst_row_offsets[inst + 1];
      for (int i = b + tid; i < e; i += blockDim.x) {
        const int row = cat.inst_rows[i];
        const double p = pcol[row];
        const int zn = cat.zone_id[row];
        if (p == p && zn != SKYOPT_NONE16 && zn < max_zones) bprice[zn] = p;
      }
    }
  } else {
    const int b = cat.inst_row_offsets[inst], e = cat.inst_row_offsets[inst + 1];
    for (int i = b + tid; i < e; i += blockDim.x) push_row(cat.inst_rows[i]);
  }
  __syncthreads();
  if (s_n > sort_n) {
    if (tid == 0) { atomicExch(err_flag, 1); out.slot_count[s] = 0; out.slot_inst[s] = inst; }
    return;
  }
  const int n = s_n;
  // sort_values([price, Region, AvailabilityZone]) -- ids are ranks in string
  // order, the row id keeps equal keys in CSV order.
  sort_pairs(k1, k2, s_t1, s_t2, n, sort_n);
  for (int i = tid; i < n; i += blockDim.x) {
    const int rg = (int)(k2[i] >> 48);
    atomicMin(&first_pos[rg], i);
  }
  __syncthreads();

  // Second key: [us regions first,] region first-appearance, sorted position.
  // Each thread rewrites only its own entries: k1 <- ordering key (or "none"
  // when the entry is filtered out), k2 <- catalog row.
  for (int i = tid; i < sort_n; i += blockDim.x) {
    uint64_t key = kKeyNone, payload = kKeyNone;
    if (i < n) {
      const uint64_t v = k2[i];
      const int rg = (int)(v >> 48);
      const int zn = (int)((v >> 32) & 0xFFFF);
      bool keep = true;
      if (S.region_id >= 0 && rg != S.region_id) keep = false;
      if (S.region_set >= 0 &&
          !test_bit(acc_sets + (int64_t)S.region_set * SKYOPT_ACC_SET_WORDS, (uint32_t)rg & 1023u))
        keep = false;  // image_id / ssh_proxy_command region allow-list
      if (S.zone_id >= 0 && (!has_zones || zn != S.zone_id)) keep = false;
      const bool split = S.split_by_zone && has_zones;
      // Region-level candidates: the region's first sorted row carries its
      // min price. With an explicit zone the (single) matching row is kept.
      if (!split && S.zone_id < 0 && first_pos[rg] != i) keep = false;
      if (gcp_acc && inst >= 0) {
        const double hb = (zn < max_zones) ? bprice[zn] : kNaN;
        if (hb != hb) keep = false;
      }
      if (keep) {
        const uint64_t us = (S.us_first && !cat.region_is_us[reg0 + rg]) ? 1 : 0;
        key = (us << 48) | ((uint64_t)first_pos[rg] << 24) | (uint64_t)i;
        payload = (uint64_t)(uint32_t)(v & 0xFFFFFFFFu);
      }
    }
    k1[i] = key;
    // filtered-out entries keep distinct (none, i) pairs: the counting sort
    // needs unique keys
    k2[i] = (key == kKeyNone && i < n) ? (uint64_t)i : payload;
  }
  sort_pairs(k1, k2, s_t1, s_t2, n, sort_n);

  const int64_t off = slot_off[s];
  int count = 0;
  for (int i = tid; i < sort_n; i += blockDim.x) {
    if (k1[i] == kKeyNone) continue;
    const int row = (int)(k2[i] & 0xFFFFFFFFu);
    const int rg = cat.region_id[row];
    const int zn = cat.zone_id[row];
    const bool split = S.split_by_zone && has_zones;
    out.cand_region[off + i] = rg;
    out.cand_zone[off + i] = (split || S.zone_id >= 0) ? (has_zones ? zn : -1) : -1;
    double pa = pcol[row], pb = 0.0;
    if (gcp_acc) {
      // accelerator price at this zone: SpotPrice, falling back to Price when
      // spot is NaN (gcp_catalog.py:433-442); host VM price from group B.
      pb = pa;
      pa = (inst >= 0) ? bprice[zn] : 0.0;
    }
    out.cand_price_a[off + i] = pa;
    out.cand_price_b[off + i] = pb;
  }
  // count = number of valid keys (they are sorted to the front)
  __syncthreads();
  if (tid == 0) {
    int lo = 0, hi = sort_n;
    while (lo < hi) { int mid = (lo + hi) >> 1; if (k1[mid] != kKeyNone) lo = mid + 1; else hi = mid; }
    count = lo;
    out.slot_count[s] = count;
    out.slot_inst[s] = inst;
  }
}


// ---------------------------------------------------------------------------
// K3: one block per DAG.
constexpr int kSolveThreads = 1024;  // 32 warps: one per task of a short chain
constexpr int kMaxDagTasks = 16;  // exact search only; chains are unbounded
constexpr int kFastTasks = 32;    // chain DP kept in shared memory
constexpr int kDpCap = 1024;      // ... when every task has <= kDpCap candidates

struct SolveIn {
  const SkyoptSlot *slots;
  const SkyoptTask *tasks;
  const int32_t *parents;
  const double *tariffs;
  const SkyoptBlocked *blocked;
  const SkyoptDag *dags;
  const int64_t *slot_off;   // [n_slots] into the expand candidate buffers
  const int64_t *task_off;   // [n_tasks+1] into the task candidate arrays
  ExpandOut ex;
  int tables_only;           // candidates were given by the caller: no slots
  const SkyoptReservation *res;  // reserved capacity table (skyopt_reserve.cuh)
  int32_t n_res;                 // 0 = none: values are hourly * hours * num_nodes
};

struct SolveWork {
  int32_t *tc_ref;    // index into the expand candidate buffers
  int32_t *tc_slot;
  int32_t *tc_cloud;
  double *tc_hourly;
  double *tc_value;
  double *dp;
  int32_t *back;
};

struct SolveOut {
  SkyoptCandidate *chosen;     // [n_tasks]
  int32_t *chosen_index;       // [n_tasks]
  int32_t *task_n;             // [n_tasks]
  SkyoptDagResult *dag;        // [n_dags]
  unsigned long long *trace;   // SKYOPT_TRACE timeline (kernel 2), or null
};

__device__ __forceinline__ void lexmin(double &v, int &i, double ov, int oi) {
  if (ov < v || (ov == v && oi < i)) { v = ov; i = oi; }
}

// K3a: one block per task -- its candidates in the reference's order
// (requested Resources -> enabled clouds -> region/zone order), minus the
// blocked ones, with their cost / time value.
constexpr int kGatherThreads = 128;
constexpr int kMaxTaskSlots = 64;

__global__ void __launch_bounds__(kGatherThreads)
gather_kernel(CatDev cat, SolveIn in, SolveWork w, const int32_t *__restrict__ task_dag,
              int32_t *__restrict__ task_n) {
  constexpr int kWarps = kGatherThreads / 32;
  __shared__ int s_cnt[kMaxTaskSlots + 1];   // exclusive prefix of slot counts
  __shared__ int s_inst[kMaxTaskSlots];
  __shared__ int s_acc[kMaxTaskSlots];
  __shared__ int s_wcount[kWarps];
  __shared__ int s_pos;
  const int t = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const SkyoptTask TK = in.tasks[t];
  const SkyoptDag D = in.dags[task_dag[t]];
  const int64_t toff = in.task_off[t];
  const int n_slots = TK.slot_end - TK.slot_begin;
  int kept_total = 0;
  for (int s0 = 0; s0 < n_slots; s0 += kMaxTaskSlots) {
    const int ns = min(kMaxTaskSlots, n_slots - s0);
    if (tid < ns) {
      const int s = TK.slot_begin + s0 + tid;
      const int inst = in.ex.slot_inst[s];
      int acc = in.slots[s].cand_acc_key;
      if (acc < 0 && inst >= 0) acc = cat.inst_acc_key[inst];
      s_inst[tid] = inst;
      s_acc[tid] = acc;
      s_cnt[tid + 1] = in.ex.slot_count[s];
    }
    if (tid == 0) { s_cnt[0] = 0; s_pos = kept_total; }
    __syncthreads();
    if (tid == 0) for (int i = 0; i < ns; ++i) s_cnt[i + 1] += s_cnt[i];
    __syncthreads();
    const int total = s_cnt[ns];
    for (int base = 0; base < total; base += kGatherThreads) {
      const int g = base + tid;
      bool keep = g < total;
      int ls = 0, i = 0, s = 0, rg = 0, zn = -1;
      double hourly = 0.0, value = 0.0;
      int64_t ref = 0;
      if (keep) {
        while (s_cnt[ls + 1] <= g) ++ls;
        i = g - s_cnt[ls];
        s = TK.slot_begin + s0 + ls;
        const SkyoptSlot S = in.slots[s];
        ref = in.slot_off[s] + i;
        rg = in.ex.cand_region[ref];
        zn = in.ex.cand_zone[ref];
        const int inst = s_inst[ls], cand_acc = s_acc[ls];
        for (int b = D.blocked_begin; b < D.blocked_end; ++b) {
          const SkyoptBlocked B = in.blocked[b];
          const bool m = (B.cloud == -1 || B.cloud == S.cloud) &&
                         (B.inst_id == -1 || B.inst_id == inst) &&
                         (B.region_id == -1 || B.region_id == rg) &&
                         (B.zone_id == -1 || B.zone_id == zn) &&
                         (B.acc_key == -1 || B.acc_key == cand_acc) &&
                         (B.use_spot == -1 || B.use_spot == S.use_spot);
          if (m) { keep = false; break; }
        }
        // float(hourly_cost * hours) * max(num_nodes - reserved, 0); spot
        // and zone-less candidates have no reserved nodes
        hourly = __dadd_rn(in.ex.cand_price_a[ref], in.ex.cand_price_b[ref]);
        double mult = S.node_mult;
        if (in.n_res && D.minimize_cost && !S.use_spot && zn >= 0 && inst >= 0)
          mult = reserved_node_mult(mult, reserved_nodes(in.res, in.n_res, S.cloud, inst, zn));
        value = D.minimize_cost
                    ? __dmul_rn(__dmul_rn(hourly, S.hours), mult)
                    : S.time_value;
        if (keep) {
          // stash the cloud in the low bits of nothing: written below
        }
      }
      const uint32_t bal = __ballot_sync(0xFFFFFFFFu, keep);
      if (lane == 0) s_wcount[warp] = __popc(bal);
      __syncthreads();
      int prefix = s_pos;
      for (int k = 0; k < warp; ++k) prefix += s_wcount[k];
      if (keep) {
        const int64_t o = toff + prefix + __popc(bal & ((1u << lane) - 1u));
        w.tc_ref[o] = (int32_t)ref;
        w.tc_slot[o] = s;
        w.tc_cloud[o] = in.slots[s].cloud;
        w.tc_hourly[o] = hourly;
        w.tc_value[o] = value;
      }
      __syncthreads();
      if (tid == 0) {
        int tot = 0;
        for (int k = 0; k < kWarps; ++k) tot += s_wcount[k];
        s_pos += tot;
      }
      __syncthreads();
    }
    kept_total = s_pos;
    __syncthreads();
  }
  if (tid == 0) task_n[t] = kept_total;
}

__device__ __forceinline__ void solve_mark(const SolveOut &out, int slot) {
  if (out.trace && threadIdx.x == 0 && blockIdx.x < 4096)
    out.trace[((size_t)2 * 4096 + blockIdx.x) * 16 + slot] = global_ns();
}

__global__ void __launch_bounds__(kSolveThreads)
solve_kernel(CatDev cat, SolveIn in, SolveWork w, SolveOut out) {
  constexpr int kWarps = kSolveThreads / 32;
  __shared__ int s_fail;
  __shared__ double s_best_val[SKYOPT_MAX_CLOUDS];
  __shared__ int s_best_idx[SKYOPT_MAX_CLOUDS];
  __shared__ double s_tb_val[kMaxDagTasks][SKYOPT_MAX_CLOUDS];
  __shared__ int s_tb_idx[kMaxDagTasks][SKYOPT_MAX_CLOUDS];
  __shared__ int s_opt[kMaxDagTasks][SKYOPT_MAX_CLOUDS];  // cloud options
  __shared__ int s_nopt[kMaxDagTasks];
  __shared__ double s_red_val[kWarps];
  __shared__ long long s_red_idx[kWarps];

  solve_mark(out, 0);
  const SkyoptDag D = in.dags[blockIdx.x];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int C = cat.n_clouds;
  const int T = D.task_end - D.task_begin;
  if (tid == 0) s_fail = -1;
  __syncthreads();

  // ---- Phase A ran in gather_kernel: candidate tables are ready. First
  // task without a candidate (all tasks are checked at once: a serial scan
  // would be one dependent memory round trip per task).
  __shared__ int s_first_empty;
  if (tid == 0) s_first_empty = 0x7FFFFFFF;
  __syncthreads();
  for (int lt = tid; lt < T; lt += kSolveThreads)
    if (out.task_n[D.task_begin + lt] == 0) atomicMin(&s_first_empty, lt);
  __syncthreads();
  if (tid == 0 && s_first_empty != 0x7FFFFFFF) s_fail = s_first_empty;
  __syncthreads();
  if (s_fail >= 0) {
    if (tid == 0) {
      SkyoptDagResult r; r.status = 1; r.task_fail = s_fail;
      r.objective = __longlong_as_double(0x7FF8000000000000ll);
      out.dag[blockIdx.x] = r;
    }
    return;
  }

  const double kInf = __longlong_as_double(0x7FF0000000000000ll);
  solve_mark(out, 1);

  // ---- Phase B, fast path for chains of up to kFastTasks tasks. The
  // recurrence  dp[c] = value[c] + min_p (dp[p] + egress(p, c))  is the
  // reference's (optimizer.py:456-470), but it is not evaluated task after
  // task: egress depends on the two clouds only and x -> fl(x + e) is
  // monotone, so with  mv[t][g] = min value of task t's candidates in cloud g
  // (all tasks at once) the per-cloud minima of dp obey a recurrence over
  // C-vectors,
  //   B[t][h] = min_g fl(D[t-1][g] + e_t(g, h)),  D[t][g] = fl(mv[t][g] + B[t][g]),
  // which one warp walks in shared memory; the winners (first minimum in
  // candidate order, as the strict '<' of the reference picks) are then found
  // for all (task, child cloud) pairs in parallel from the same sums the
  // reference forms. Three barriers instead of two per task.
  {
    __shared__ int s_tn[kFastTasks], s_src[kFastTasks], s_np[kFastTasks];
    __shared__ long long s_toff[kFastTasks];
    __shared__ double s_tar[kFastTasks][SKYOPT_MAX_CLOUDS];
    __shared__ unsigned long long s_mv[kFastTasks][SKYOPT_MAX_CLOUDS];  // price_key(min value)
    __shared__ double s_B[kFastTasks][SKYOPT_MAX_CLOUDS];
    __shared__ double s_D[kFastTasks][SKYOPT_MAX_CLOUDS];
    __shared__ int s_bk_idx[kFastTasks + 1][SKYOPT_MAX_CLOUDS];
    __shared__ unsigned char s_bk_cl[kFastTasks + 1][SKYOPT_MAX_CLOUDS];
    __shared__ double s_obj;
    __shared__ int s_fast;
    if (tid == 0) s_fast = (D.is_chain && T <= kFastTasks) ? 1 : 0;
    __syncthreads();
    if (s_fast) {
      if (tid < T) {
        const int t = D.task_begin + tid;
        const SkyoptTask TK = in.tasks[t];
        s_tn[tid] = out.task_n[t];
        s_toff[tid] = in.task_off[t];
        s_np[tid] = TK.n_parents;
        s_src[tid] = TK.n_parents ? TK.edge_tariff_begin : TK.src_tariff_begin;
      }
      for (int i = tid; i < T * C; i += kSolveThreads) s_mv[i / C][i % C] = kKeyNone;
      __syncthreads();
      for (int i = tid; i < T * C; i += kSolveThreads) {
        const int lt = i / C, cc = i % C;
        s_tar[lt][cc] = s_src[lt] >= 0 ? in.tariffs[s_src[lt] + cc] : 0.0;
      }
      // per-(task, cloud) minimum value, every task at once (a warp per task)
      for (int lt = warp; lt < T; lt += kWarps) {
        const int n = s_tn[lt];
        const long long toff = s_toff[lt];
        for (int c = lane; c < n; c += 32)
          atomicMin(&s_mv[lt][w.tc_cloud[toff + c]], (unsigned long long)price_key(w.tc_value[toff + c]));
      }
      __syncthreads();
      solve_mark(out, 2);
      if (warp == 0) {
        // the C-vector recurrence: lane h owns cloud h
        for (int lt = 0; lt < T; ++lt) {
          if (lane < C) {
            double b;
            if (s_np[lt] == 0) {
              b = s_tar[lt][lane];  // dummy source: 0 + egress from the inputs' cloud
            } else {
              b = kInf;
              for (int g = 0; g < C; ++g) {
                const double e = (g != lane) ? s_tar[lt][g] : 0.0;
                const double v = __dadd_rn(s_D[lt - 1][g], e);
                if (v < b) b = v;
              }
            }
            s_B[lt][lane] = b;
            const unsigned long long mk = s_mv[lt][lane];
            s_D[lt][lane] = (mk == kKeyNone) ? kInf : __dadd_rn(key_price(mk), b);
          }
          __syncwarp();
        }
      }
      __syncthreads();
      solve_mark(out, 3);
      // winners: pair (lt, h) = first minimum over task lt's candidates p of
      // fl(dp[p] + e_{lt+1}(cloud(p), h)); the pair (T-1, 0) is the dummy sink
      // (egress 0).
      const int n_pairs = (T - 1) * C + 1;
      for (int pr = warp; pr < n_pairs; pr += kWarps) {
        const bool sink = pr == n_pairs - 1;
        const int lt = sink ? T - 1 : pr / C;    // parent task
        const int h = sink ? 0 : pr % C;         // child cloud
        double bv = kInf; int bi = 0x7FFFFFFF;
        // a child cloud without candidates never asks for its parent
        if (sink || s_mv[lt + 1][h] != kKeyNone) {
          const int n = s_tn[lt];
          const long long toff = s_toff[lt];
          for (int p = lane; p < n; p += 32) {
            const int cp = w.tc_cloud[toff + p];
            const double dpp = __dadd_rn(w.tc_value[toff + p], s_B[lt][cp]);
            const double e = (!sink && cp != h) ? s_tar[lt + 1][cp] : 0.0;
            lexmin(bv, bi, sink ? dpp : __dadd_rn(dpp, e), p);
          }
          for (int o = 16; o; o >>= 1) {
            const double ov = __shfl_xor_sync(0xFFFFFFFFu, bv, o);
            const int oi = __shfl_xor_sync(0xFFFFFFFFu, bi, o);
            lexmin(bv, bi, ov, oi);
          }
        }
        if (lane == 0) {
          const int slot_t = sink ? T : lt + 1;  // indexed by the child task
          s_bk_idx[slot_t][h] = bi;
          s_bk_cl[slot_t][h] = (bi != 0x7FFFFFFF) ? (unsigned char)w.tc_cloud[s_toff[lt] + bi] : 0;
          if (sink) s_obj = bv;
        }
      }
      __syncthreads();
      solve_mark(out, 4);
      if (tid == 0) {
        SkyoptDagResult r; r.status = 0; r.task_fail = -1; r.objective = s_obj;
        out.dag[blockIdx.x] = r;
        int idx = s_bk_idx[T][0];
        int cl = s_bk_cl[T][0];
        for (int lt = T - 1; lt >= 0; --lt) {
          out.chosen_index[D.task_begin + lt] = idx;
          if (lt > 0) {
            const int ni = s_bk_idx[lt][cl];
            cl = s_bk_cl[lt][cl];
            idx = ni;
          }
        }
      }
    }
    if (s_fast) goto plan_records;
  }
  if (D.is_chain) {
    // ---- Phase B: dp[c] = value[c] + min_p (dp[p] + egress(p, c)); strict
    // '<' => first minimum in candidate order (optimizer.py:456-470). The
    // egress term depends on the clouds only, so the inner minimum is taken
    // once per child cloud -- same additions, same comparisons, same winner.
    for (int t = D.task_begin; t < D.task_end; ++t) {
      const SkyoptTask TK = in.tasks[t];
      const int64_t toff = in.task_off[t];
      const int n = out.task_n[t];
      if (TK.n_parents == 0) {
        if (tid < C) {
          // parent = dummy source: 0 + egress from the inputs' cloud
          s_best_val[tid] = TK.src_tariff_begin >= 0 ? in.tariffs[TK.src_tariff_begin + tid] : 0.0;
          s_best_idx[tid] = 0;
        }
      } else {
        const int tp = D.task_begin + in.parents[TK.parent_begin];
        const int64_t poff = in.task_off[tp];
        const int np = out.task_n[tp];
        const double *tar = in.tariffs + TK.edge_tariff_begin;
        for (int cc = warp; cc < C; cc += kWarps) {
          double bv = kInf; int bi = 0x7FFFFFFF;
          for (int p = lane; p < np; p += 32) {
            const int cp = w.tc_cloud[poff + p];
            const double eg = (cp != cc) ? tar[cp] : 0.0;
            lexmin(bv, bi, __dadd_rn(w.dp[poff + p], eg), p);
          }
          for (int o = 16; o; o >>= 1) {
            const double ov = __shfl_xor_sync(0xFFFFFFFFu, bv, o);
            const int oi = __shfl_xor_sync(0xFFFFFFFFu, bi, o);
            lexmin(bv, bi, ov, oi);
          }
          if (lane == 0) { s_best_val[cc] = bv; s_best_idx[cc] = bi; }
        }
      }
      __syncthreads();
      for (int c = tid; c < n; c += kSolveThreads) {
        const int cc = w.tc_cloud[toff + c];
        w.dp[toff + c] = __dadd_rn(w.tc_value[toff + c], s_best_val[cc]);
        w.back[toff + c] = s_best_idx[cc];
      }
      __syncthreads();
    }
    // sink: 0 + min_p dp[p] (egress to the dummy sink is 0)
    {
      const int t = D.task_end - 1;
      const int64_t toff = in.task_off[t];
      const int n = out.task_n[t];
      double bv = kInf; int bi = 0x7FFFFFFF;
      for (int p = tid; p < n; p += kSolveThreads) lexmin(bv, bi, w.dp[toff + p], p);
      for (int o = 16; o; o >>= 1) {
        const double ov = __shfl_xor_sync(0xFFFFFFFFu, bv, o);
        const int oi = __shfl_xor_sync(0xFFFFFFFFu, bi, o);
        lexmin(bv, bi, ov, oi);
      }
      if (lane == 0) { s_red_val[warp] = bv; s_red_idx[warp] = bi; }
      __syncthreads();
      if (tid == 0) {
        for (int k = 1; k < kWarps; ++k) lexmin(bv, bi, s_red_val[k], (int)s_red_idx[k]);
        SkyoptDagResult r; r.status = 0; r.task_fail = -1; r.objective = bv;
        out.dag[blockIdx.x] = r;
        int idx = bi;
        for (int tt = D.task_end - 1; tt >= D.task_begin; --tt) {
          out.chosen_index[tt] = idx;
          idx = w.back[in.task_off[tt] + idx];
        }
      }
    }
  } else {
    // ---- Phase B': exact search replacing the PuLP/CBC ILP
    // (optimizer.py:490-637). Egress depends on (cloud_u, cloud_v) only, so
    // within one cloud the cheapest candidate of a task dominates; what is
    // left is an exhaustive enumeration of cloud assignments.
    if (T > kMaxDagTasks) {
      if (tid == 0) {
        SkyoptDagResult r; r.status = 2; r.task_fail = -1;
        r.objective = __longlong_as_double(0x7FF8000000000000ll);
        out.dag[blockIdx.x] = r;
      }
      return;
    }
    for (int lt = warp; lt < T; lt += kWarps) {
      const int t = D.task_begin + lt;
      const int64_t toff = in.task_off[t];
      const int n = out.task_n[t];
      for (int cc = 0; cc < C; ++cc) {
        double bv = kInf; int bi = 0x7FFFFFFF;
        for (int p = lane; p < n; p += 32)
          if (w.tc_cloud[toff + p] == cc) lexmin(bv, bi, w.tc_value[toff + p], p);
        for (int o = 16; o; o >>= 1) {
          const double ov = __shfl_xor_sync(0xFFFFFFFFu, bv, o);
          const int oi = __shfl_xor_sync(0xFFFFFFFFu, bi, o);
          lexmin(bv, bi, ov, oi);
        }
        if (lane == 0) { s_tb_val[lt][cc] = bv; s_tb_idx[lt][cc] = bi; }
      }
      __syncwarp();
      if (lane == 0) {
        // options ordered by the candidate index of their representative
        int no = 0;
        for (int cc = 0; cc < C; ++cc)
          if (s_tb_idx[lt][cc] != 0x7FFFFFFF) s_opt[lt][no++] = cc;
        for (int a = 1; a < no; ++a) {
          const int v = s_opt[lt][a]; int b2 = a - 1;
          while (b2 >= 0 && s_tb_idx[lt][s_opt[lt][b2]] > s_tb_idx[lt][v]) { s_opt[lt][b2 + 1] = s_opt[lt][b2]; --b2; }
          s_opt[lt][b2 + 1] = v;
        }
        s_nopt[lt] = no;
      }
    }
    __syncthreads();
    long long total = 1;
    bool too_big = false;
    for (int lt = 0; lt < T; ++lt) {
      total *= s_nopt[lt];
      if (total > (1ll << 26)) { too_big = true; break; }  // ~10 ms of one block; beyond: status 2
    }
    if (too_big) {
      if (tid == 0) {
        SkyoptDagResult r; r.status = 2; r.task_fail = -1;
        r.objective = __longlong_as_double(0x7FF8000000000000ll);
        out.dag[blockIdx.x] = r;
      }
      return;
    }
    double bv = kInf; long long bid = 0x7FFFFFFFFFFFFFFFll;
    for (long long id = tid; id < total; id += kSolveThreads) {
      int cl[kMaxDagTasks];
      long long rem = id;
      for (int lt = T - 1; lt >= 0; --lt) {  // task 0 = most significant digit
        const int no = s_nopt[lt];
        cl[lt] = s_opt[lt][(int)(rem % no)];
        rem /= no;
      }
      double obj;
      if (D.minimize_cost) {
        obj = 0.0;
        for (int lt = 0; lt < T; ++lt) obj = __dadd_rn(obj, s_tb_val[lt][cl[lt]]);
        for (int lt = 0; lt < T; ++lt) {
          const SkyoptTask TK = in.tasks[D.task_begin + lt];
          if (TK.n_parents == 0 && TK.src_tariff_begin >= 0)
            obj = __dadd_rn(obj, in.tariffs[TK.src_tariff_begin + cl[lt]]);
          for (int k = 0; k < TK.n_parents; ++k) {
            const int lp = in.parents[TK.parent_begin + k];
            if (cl[lp] != cl[lt])
              obj = __dadd_rn(obj, in.tariffs[TK.edge_tariff_begin + k * C + cl[lp]]);
          }
        }
      } else {
        double fin[kMaxDagTasks];
        obj = 0.0;
        for (int lt = 0; lt < T; ++lt) {
          const SkyoptTask TK = in.tasks[D.task_begin + lt];
          double start = 0.0;
          if (TK.n_parents == 0 && TK.src_tariff_begin >= 0)
            start = fmax(start, in.tariffs[TK.src_tariff_begin + cl[lt]]);
          for (int k = 0; k < TK.n_parents; ++k) {
            const int lp = in.parents[TK.parent_begin + k];
            const double eg = (cl[lp] != cl[lt])
                                  ? in.tariffs[TK.edge_tariff_begin + k * C + cl[lp]] : 0.0;
            start = fmax(start, __dadd_rn(fin[lp], eg));
          }
          fin[lt] = __dadd_rn(s_tb_val[lt][cl[lt]], start);
          obj = fmax(obj, fin[lt]);  // sink waits for every leaf
        }
      }
      if (obj < bv || (obj == bv && id < bid)) { bv = obj; bid = id; }
    }
    for (int o = 16; o; o >>= 1) {
      const double ov = __shfl_xor_sync(0xFFFFFFFFu, bv, o);
      const long long oi = __shfl_xor_sync(0xFFFFFFFFu, bid, o);
      if (ov < bv || (ov == bv && oi < bid)) { bv = ov; bid = oi; }
    }
    if (lane == 0) { s_red_val[warp] = bv; s_red_idx[warp] = bid; }
    __syncthreads();
    if (tid == 0) {
      for (int k = 1; k < kWarps; ++k)
        if (s_red_val[k] < bv || (s_red_val[k] == bv && s_red_idx[k] < bid)) { bv = s_red_val[k]; bid = s_red_idx[k]; }
      SkyoptDagResult r; r.status = 0; r.task_fail = -1; r.objective = bv;
      out.dag[blockIdx.x] = r;
      long long rem = bid;
      for (int lt = T - 1; lt >= 0; --lt) {
        const int no = s_nopt[lt];
        const int cc = s_opt[lt][(int)(rem % no)];
        rem /= no;
        out.chosen_index[D.task_begin + lt] = s_tb_idx[lt][cc];
      }
    }
  }
plan_records:
  __syncthreads();
  solve_mark(out, 5);
  if (in.tables_only) return;
  // ---- the plan as candidate records
  for (int lt = tid; lt < T; lt += kSolveThreads) {
    const int t = D.task_begin + lt;
    const int64_t o = in.task_off[t] + out.chosen_index[t];
    const int64_t ref = w.tc_ref[o];
    const int s = w.tc_slot[o];
    SkyoptCandidate c;
    c.slot = s;
    c.inst_id = in.ex.slot_inst[s];
    c.region_id = in.ex.cand_region[ref];
    c.zone_id = in.ex.cand_zone[ref];
    c.hourly = w.tc_hourly[o];
    c.value = w.tc_value[o];
    out.chosen[t] = c;
  }
  solve_mark(out, 6);
}

// Optional full candidate tables (display / _fill_in_launchable_resources).
__global__ void table_kernel(SolveIn in, SolveWork w, const int32_t *task_n,
                             int n_tasks, const int64_t *__restrict__ out_off,
                             SkyoptCandidate *__restrict__ table) {
  const int t = blockIdx.x;
  if (t >= n_tasks) return;
  const int n = task_n[t];
  const int64_t toff = in.task_off[t];
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int64_t o = toff + i;
    const int64_t ref = w.tc_ref[o];
    const int s = w.tc_slot[o];
    SkyoptCandidate c;
    c.slot = s;
    c.inst_id = in.ex.slot_inst[s];
    c.region_id = in.ex.cand_region[ref];
    c.zone_id = in.ex.cand_zone[ref];
    c.hourly = w.tc_hourly[o];
    c.value = w.tc_value[o];
    table[out_off[t] + i] = c;
  }
}

// Evict the catalog from L2 between timed iterations (bench.py).
// Cheapest offering of each group (an instance type's rows, or -- GCP -- the
// accelerator-only rows of one (name, count) key): the row with the
// lexicographically smallest (Price, SpotPrice), missing values last, first
// CSV row on ties -- what list_accelerators_impl keeps after
// sort_values(['Price', 'SpotPrice'[, 'Region']]).drop_duplicates(keep='first')
// (common.py:756-768) -- over the regions the caller's filter allows; with
// `per_region` one winner per region. One block per group; three passes over
// the group's rows with shared-memory atomics (price, then spot price among
// the cheapest, then row).
__global__ void __launch_bounds__(128)
offer_kernel(CatDev cat, int cloud, int by_acc_key, const int32_t *__restrict__ group_ids,
             const uint32_t *__restrict__ region_mask, int per_region, int n_regions,
             int32_t *__restrict__ out_rows) {
  extern __shared__ unsigned long long offer_smem[];
  const int slots = per_region ? n_regions : 1;
  unsigned long long *best_p = offer_smem;          // [slots]
  unsigned long long *best_s = best_p + slots;      // [slots]
  unsigned int *best_row = reinterpret_cast<unsigned int *>(best_s + slots);  // [slots]
  const int g = group_ids[blockIdx.x];
  const int tid = threadIdx.x;
  for (int i = tid; i < slots; i += blockDim.x) { best_p[i] = kKeyNone; best_s[i] = kKeyNone; best_row[i] = kRowNone; }
  __syncthreads();
  const int32_t *rows = by_acc_key ? cat.acc_rows : cat.inst_rows;
  const int32_t *offs = by_acc_key ? cat.acc_row_offsets : cat.inst_row_offsets;
  const int b = offs[g], e = offs[g + 1];
  const int r0 = cat.cloud_row_offsets[cloud], r1 = cat.cloud_row_offsets[cloud + 1];
  auto allowed = [&](int row, int &slot) {
    if (row < r0 || row >= r1) return false;
    const int rg = cat.region_id[row];
    if (region_mask && !((region_mask[rg >> 5] >> (rg & 31)) & 1u)) return false;
    slot = per_region ? rg : 0;
    return true;
  };
  auto keys = [&](int row, unsigned long long &pk, unsigned long long &sk) {
    const double p = cat.price[row], sp = cat.spot[row];
    pk = (p == p) ? price_key(p) : kKeyNaN;
    sk = (sp == sp) ? price_key(sp) : kKeyNaN;
  };
  for (int i = b + tid; i < e; i += blockDim.x) {
    const int row = rows[i]; int slot;
    if (!allowed(row, slot)) continue;
    unsigned long long pk, sk; keys(row, pk, sk);
    atomicMin(&best_p[slot], pk);
  }
  __syncthreads();
  for (int i = b + tid; i < e; i += blockDim.x) {
    const int row = rows[i]; int slot;
    if (!allowed(row, slot)) continue;
    unsigned long long pk, sk; keys(row, pk, sk);
    if (pk == best_p[slot]) atomicMin(&best_s[slot], sk);
  }
  __syncthreads();
  for (int i = b + tid; i < e; i += blockDim.x) {
    const int row = rows[i]; int slot;
    if (!allowed(row, slot)) continue;
    unsigned long long pk, sk; keys(row, pk, sk);
    if (pk == best_p[slot] && sk == best_s[slot]) atomicMin(&best_row[slot], (unsigned int)row);
  }
  __syncthreads();
  for (int i = tid; i < slots; i += blockDim.x)
    out_rows[(int64_t)blockIdx.x * slots + i] = (best_row[i] == kRowNone) ? -1 : (int32_t)best_row[i];
}

__global__ void flush_kernel(uint32_t *buf, int64_t n, uint32_t v) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    buf[i] = v + (uint32_t)i;
}

// Second half of the optional write-then-read flush: after this pass the L2
// holds clean lines only, so evictions inside the timed region are not
// write-backs of the flush's own data.
__global__ void flush_read_kernel(const uint32_t *buf, int64_t n, uint32_t *sink) {
  uint32_t acc = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    acc ^= __ldcg(buf + i);
  if (acc == 0x9E3779B9u) *sink = acc;  // keeps the loads alive
}

}  // namespace skyopt
