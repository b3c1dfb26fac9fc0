// skyopt_fast.cuh -- the round-2 hot path: a bit-parallel streaming scan and
// the fused expansion / blocked filter / cost kernel.
//
// K1' scan2_kernel  Same answers as scan_kernel (reference
//                   sky/catalog/common.py:518-569, :641-694), different
//                   algorithm. At ingest every row is reduced to three small
//                   dictionary codes -- (vCPUs, MemoryGiB), (flags, accelerator
//                   key, local disk) and (region, zone) -- and to its RANK in
//                   the cloud's (price, row) order, one layout per price column,
//                   10 bytes per row, each 128-row chunk stored in ascending
//                   rank. A block evaluates the (at most 32) fused constraint
//                   vectors of its group once per dictionary ENTRY into three
//                   shared-memory tables of 32-bit masks (bit q = query q
//                   accepts the entry). A row then costs three table look-ups
//                   and two ANDs for all 32 queries at once; a 32x32 bit
//                   transpose over the warp (five shuffles) hands lane q the
//                   set of lanes whose rows query q accepts, and because lanes
//                   hold ascending ranks the first set bit is the chunk's
//                   argmin. No fp64 in the streaming loop, no per-(row, query)
//                   work: the loop is bound by the HBM stream.
// K2' place_kernel  expand_kernel + gather_kernel in one launch, block per
//                   task. The (price, region, zone) ordering of an instance
//                   type's rows (common.py:793-809; resources_utils.py:454-502)
//                   does not depend on the request, so it is computed at ingest;
//                   a slot is then a filtered copy of a static list.
#pragma once

#include "skyopt_kernels.cuh"

namespace skyopt {

constexpr uint32_t kRankNone = 0xFFFFFFFFu;
constexpr int kFastWarps = kScanThreads / 32;
constexpr int kFastMaxZones = 512;      // per-warp host-VM zone table (GCP)
constexpr int kFastMaxTaskSlots = 64;
constexpr int kInlineGroups2 = 24;      // scan groups that travel in the kernel parameters

// Device-side timeline (SKYOPT_TRACE=<file>): 16 slots per block and kernel.
constexpr int kTraceSlots = 16;
constexpr int kTraceBlocks = 4096;
__device__ __forceinline__ void trace_mark(unsigned long long *trace, int kernel, int slot) {
  if (trace && threadIdx.x == 0 && blockIdx.x < kTraceBlocks)
    trace[((size_t)kernel * kTraceBlocks + blockIdx.x) * kTraceSlots + slot] = global_ns();
}
__device__ __forceinline__ void trace_put(unsigned long long *trace, int kernel, int slot,
                                          unsigned long long v) {
  if (trace && blockIdx.x < kTraceBlocks)
    trace[((size_t)kernel * kTraceBlocks + blockIdx.x) * kTraceSlots + slot] = v;
}

// rank -> what the expansion needs of the cheapest row: its price (the cap
// test), its instance type and where that type's static list lives
struct RankRec {
  double price;
  int32_t row;
  int32_t inst;
  int32_t list_off;  // = inst_list[inst] (one dependent load less)
  int32_t cnt[2];
  int32_t acc_key;
};
static_assert(sizeof(RankRec) == 32, "RankRec layout");

// One entry of an instance type's (or accelerator key's) static launchable
// order: rows with a price, sorted by (price, region, zone), regrouped by the
// first appearance of their region (resources_utils.py:454-502).
struct ExpEnt {
  double price;
  uint32_t row;      // bit 31: first (cheapest) row of its region
  uint16_t rg, zn;
};
static_assert(sizeof(ExpEnt) == 16, "ExpEnt layout");
constexpr uint32_t kRegionFirst = 0x80000000u;

// Where a group's static list lives (instance type / accelerator key).
struct ListRec {
  int32_t off;       // into exp_ent / aexp_ent (both price columns)
  int32_t cnt[2];    // entries kept per price column
  int32_t acc_key;   // instance types: accelerators of the type (inst_acc_key)
};
static_assert(sizeof(ListRec) == 16, "ListRec layout");

struct FastCat {
  // scan layouts, one per price column: chunk-sorted ranks and class codes
  const uint32_t *s_rank[2];
  const uint16_t *s_cm[2], *s_fa[2], *s_rz[2];
  const uint32_t *cmin[2];        // [n_rows / 128] smallest rank of the chunk
  const RankRec *rank_rec[2];     // [cloud_row_offsets[c] + rank]
  // class dictionaries, per cloud
  const double2 *cm_val;          // (vCPUs, MemoryGiB)
  const uint32_t *fa_key;         // flags | acc_key << 16
  const double *fa_disk;
  const uint32_t *rz_key;         // region | zone << 16
  // static launchable orders
  const ExpEnt *exp_ent[2];
  const ListRec *inst_list;       // [n_inst]
  const ExpEnt *aexp_ent[2];
  const ListRec *acc_list;        // [n_acc_keys]
};

struct Scan2Group {
  int32_t cloud, col;
  int32_t q_begin, q_count;       // into the scan-order query records
  int32_t n_cm, n_fa, n_rz;       // class counts of the cloud
  int32_t cm_off, fa_off, rz_off; // into the class dictionaries
  int32_t chunk0, n_chunks;       // the cloud's 128-row chunks
  int32_t piece0, n_pieces;       // the group's share of the launch's pieces
  int32_t index;                  // position in the launch's group array
  int32_t need_any;               // some query of the group wants any_stage1
};

struct Scan2Args {
  CatDev cat;
  FastCat f;
  const ScanQuery *squeries;
  const Scan2Group *groups;
  int n_groups, n_pieces;
  uint32_t *best_rank;            // [n_queries] by caller index; atomicMin
  uint32_t *any1;                 // [n_queries] any_stage1
  int32_t *zero_flag;
  uint32_t noprune;               // 1: ignore the zone map and the bound
  uint32_t force_any;             // the caller reads any_stage1 of every query
  uint32_t cap_fa, cap_cm, cap_rz;  // shared-memory capacities (entries)
  // cooperative launch only: the blocks of a group build its tables together
  // (one slice each) in `shared_tables` and wait on `group_ready`
  uint32_t *shared_tables;        // [n_groups][2 * cap_fa + cap_cm + cap_rz] or null
  unsigned int *group_ready;      // [n_groups] slices published (zero between launches)
  unsigned long long *trace;
  int32_t inline_piece0[kInlineGroups2];
  Scan2Group inline_groups[kInlineGroups2];
};

// 32x32 bit transpose over the warp: out(lane q) bit l = in(lane l) bit q.
// Five block-swap steps; in step j a lane keeps the half of its bits that
// already sits in the right block and takes the other half from lane ^ j,
// shifted by j -- as a rotation, so that both directions are one funnel shift
// and the merge one LOP3: three instructions per step. The per-lane masks and
// rotation amounts are computed once per kernel.
struct TransposeLane {
  uint32_t keep[5];
  uint32_t rot[5];
};
__device__ __forceinline__ TransposeLane transpose_lane(int lane) {
  TransposeLane t;
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    const int j = 16 >> i;
    const uint32_t m = (j == 16) ? 0x0000FFFFu : (j == 8) ? 0x00FF00FFu
                     : (j == 4) ? 0x0F0F0F0Fu : (j == 2) ? 0x33333333u : 0x55555555u;
    // lanes with bit j clear keep the bits with bit j clear and take the
    // partner's low-block bits shifted up; the others the mirror image
    t.keep[i] = (lane & j) ? ~m : m;
    t.rot[i] = (lane & j) ? (uint32_t)(32 - j) : (uint32_t)j;
  }
  return t;
}
__device__ __forceinline__ uint32_t warp_transpose32(uint32_t x, const TransposeLane &t) {
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    const uint32_t p = __shfl_xor_sync(0xFFFFFFFFu, x, 16 >> i);
    const uint32_t r = __funnelshift_l(p, p, t.rot[i]);
    x = (x & t.keep[i]) | (r & ~t.keep[i]);
  }
  return x;
}

#ifndef SKYOPT_RING_DEPTH
#define SKYOPT_RING_DEPTH 3
#endif
constexpr int kRingDepth = SKYOPT_RING_DEPTH;   // chunk slots per warp (cp.async ring)
struct RingSlot {
  uint32_t rk[kZoneRows];
  uint16_t cm[kZoneRows], fa[kZoneRows], rz[kZoneRows];
};
static_assert(sizeof(RingSlot) == 10 * kZoneRows, "ring slot = one chunk of the 10 B/row layout");

__device__ __forceinline__ void cp_async16(void *dst, const void *src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async8(void *dst, const void *src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

struct Rows2 {
  uint4 rk;       // ranks of positions 4*lane .. 4*lane+3 (ascending)
  uint2 cm, fa, rz;
};

// Loads that stay where they are written (the prologue issues the first
// chunk's rows before the tables are built).
__device__ __forceinline__ uint4 ldg_nc_v4(const void *p) {
  uint4 v;
  asm volatile("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ uint2 ldg_nc_v2(const void *p) {
  uint2 v;
  asm volatile("ld.global.nc.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
  return v;
}
__device__ __forceinline__ uint32_t ldg_nc_u32(const void *p) {
  uint32_t v;
  asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}

__device__ __forceinline__ Rows2 load_rows2(const Scan2Args &a, int col, int64_t chunk, int lane) {
  Rows2 r;
  const int64_t base = chunk * kZoneRows;
  r.rk = ldg_nc_v4(reinterpret_cast<const uint4 *>(a.f.s_rank[col] + base) + lane);
  r.cm = ldg_nc_v2(reinterpret_cast<const uint2 *>(a.f.s_cm[col] + base) + lane);
  r.fa = ldg_nc_v2(reinterpret_cast<const uint2 *>(a.f.s_fa[col] + base) + lane);
  r.rz = ldg_nc_v2(reinterpret_cast<const uint2 *>(a.f.s_rz[col] + base) + lane);
  return r;
}

// One chunk of the scan layout -> a ring slot (asynchronous, 40 B per lane).
__device__ __forceinline__ void fetch_rows2(const Scan2Args &a, int col, int64_t chunk, int lane,
                                            RingSlot &slot) {
  const int64_t base = chunk * kZoneRows + 4 * lane;
  cp_async16(slot.rk + 4 * lane, a.f.s_rank[col] + base);
  cp_async8(slot.cm + 4 * lane, a.f.s_cm[col] + base);
  cp_async8(slot.fa + 4 * lane, a.f.s_fa[col] + base);
  cp_async8(slot.rz + 4 * lane, a.f.s_rz[col] + base);
}

__device__ __forceinline__ Scan2Group find_group2(const Scan2Args &a, int p) {
  if (a.n_groups <= kInlineGroups2) {
    int idx = 0;
#pragma unroll
    for (int step = 16; step >= 1; step >>= 1) {
      const int probe = idx + step;
      if (probe < a.n_groups && probe < kInlineGroups2 && a.inline_piece0[probe] <= p) idx = probe;
    }
    return a.inline_groups[idx];
  }
  int lo = 0, hi = a.n_groups - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(&a.groups[mid].piece0) <= p) lo = mid; else hi = mid - 1;
  }
  return a.groups[lo];
}

// Shared memory of one scan2 block (dynamic): the staged constraint vectors,
// the raw class dictionaries of the cloud and the three mask tables.
struct Scan2Smem {
  ScanQuery *sq;
  uint32_t *sbest, *sany;
  uint2 *Tfa; uint32_t *Tcm, *Trz;
  double2 *d_cm; double *d_disk; uint32_t *d_fa, *d_rz;
  RingSlot *ring;   // [kFastWarps][kRingDepth]
};
__host__ __device__ inline size_t scan2_smem_bytes(size_t cap_fa, size_t cap_cm, size_t cap_rz) {
  return kQChunk * sizeof(ScanQuery) + (kQChunk + 4) * sizeof(uint32_t) +
         cap_fa * (8 + 8 + 4) + cap_cm * (4 + 16) + cap_rz * (4 + 4) + 64 +
         (size_t)kFastWarps * kRingDepth * sizeof(RingSlot);
}
__device__ __forceinline__ Scan2Smem carve_scan2(unsigned char *base, const Scan2Args &a) {
  Scan2Smem s;
  s.sq = reinterpret_cast<ScanQuery *>(base); base += kQChunk * sizeof(ScanQuery);
  s.ring = reinterpret_cast<RingSlot *>(base); base += (size_t)kFastWarps * kRingDepth * sizeof(RingSlot);
  s.d_cm = reinterpret_cast<double2 *>(base); base += (size_t)a.cap_cm * 16;
  s.Tfa = reinterpret_cast<uint2 *>(base); base += (size_t)a.cap_fa * 8;
  s.d_disk = reinterpret_cast<double *>(base); base += (size_t)a.cap_fa * 8;
  s.sbest = reinterpret_cast<uint32_t *>(base); base += kQChunk * 4;
  s.sany = reinterpret_cast<uint32_t *>(base); base += 16;
  s.Tcm = reinterpret_cast<uint32_t *>(base); base += (size_t)a.cap_cm * 4;
  s.Trz = reinterpret_cast<uint32_t *>(base); base += (size_t)a.cap_rz * 4;
  s.d_fa = reinterpret_cast<uint32_t *>(base); base += (size_t)a.cap_fa * 4;
  s.d_rz = reinterpret_cast<uint32_t *>(base);
  return s;
}

__device__ __forceinline__ void scan2_body(const Scan2Args &a, unsigned char *smem2) {
  const Scan2Smem S = carve_scan2(smem2, a);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (blockIdx.x == 0 && tid == 0 && a.zero_flag) *a.zero_flag = 0;
  trace_mark(a.trace, 0, 0);
  if (a.trace && tid == 0) {
    unsigned smid;
    asm volatile("mov.u32 %0, %smid;" : "=r"(smid));
    trace_put(a.trace, 0, 6, smid);
  }
  const bool prune = (a.noprune & 1u) == 0;
  const TransposeLane tl = transpose_lane(lane);
  uint32_t n_visit = 0, n_live = 0;

  int cur_group = -1;
  for (int p = blockIdx.x; p < a.n_pieces; p += gridDim.x) {
    const Scan2Group G = find_group2(a, p);
    const int gi = G.piece0;  // identifies the group
    const int col = G.col, nq = G.q_count;
    const int pi = p - G.piece0;
    const int chunk_begin = G.chunk0 + (int)((int64_t)G.n_chunks * pi / G.n_pieces);
    const int chunk_end = G.chunk0 + (int)((int64_t)G.n_chunks * (pi + 1) / G.n_pieces);

    // ---- this warp's chunks: chunk_begin + warp + 8 j. The summaries of its
    // first 32 chunks (one per lane) and the rows of the very first one leave
    // before anything else: they do not depend on the tables.
    const int n_mine = (chunk_end - chunk_begin - warp + kFastWarps - 1) / kFastWarps;
    RingSlot *ring = S.ring + warp * kRingDepth;
    uint4 zs = make_uint4(0, 0, 0, 0);
    uint32_t cms = 0;
    if (prune && lane < n_mine) {
      const int cl = chunk_begin + warp + kFastWarps * lane;
      zs = ldg_nc_v4(a.cat.zone_map + cl);
      cms = ldg_nc_u32(a.f.cmin[col] + cl);
    }
    __syncwarp();  // the ring's previous readers are done
    if (n_mine > 0) fetch_rows2(a, col, chunk_begin + warp, lane, ring[0]);
    cp_commit();

    if (gi != cur_group) {
      __syncthreads();  // previous group's tables are still being read
      const bool first = cur_group < 0;
      cur_group = gi;
      // ---- one round trip: constraint vectors and the cloud's dictionaries
      {
        const uint4 *src = reinterpret_cast<const uint4 *>(a.squeries + G.q_begin);
        uint4 *dst = reinterpret_cast<uint4 *>(S.sq);
        const int n16 = nq * (int)(sizeof(ScanQuery) / 16);
#pragma unroll 1
        for (int i = tid; i < n16; i += kScanThreads) dst[i] = __ldg(src + i);
#pragma unroll 1
        for (int i = tid; i < G.n_cm; i += kScanThreads) S.d_cm[i] = __ldg(a.f.cm_val + G.cm_off + i);
#pragma unroll 1
        for (int i = tid; i < G.n_fa; i += kScanThreads) {
          S.d_fa[i] = __ldg(a.f.fa_key + G.fa_off + i);
          S.d_disk[i] = __ldg(a.f.fa_disk + G.fa_off + i);
        }
#pragma unroll 1
        for (int i = tid; i < G.n_rz; i += kScanThreads) S.d_rz[i] = __ldg(a.f.rz_key + G.rz_off + i);
      }
      __syncthreads();
      trace_mark(a.trace, 0, 1);
      const long long c_tab = clock64();
      if (tid < kQChunk) {
        // a later piece starts from what the grid has found so far
        uint32_t seed = kRankNone;
        if (tid < nq && prune && !first)
          seed = *reinterpret_cast<volatile uint32_t *>(a.best_rank + S.sq[tid].qid);
        S.sbest[tid] = seed;
      }
      if (tid == 0) S.sany[0] = 0;
      // ---- the three mask tables: lane q holds query q's constraint vector in
      // registers, a warp takes one dictionary entry at a time and one ballot
      // gives the entry's 32-bit mask. Every query is evaluated on the entry
      // exactly like score_rows does on a row (same fp64 comparisons,
      // common.py:431-480). Every block of the group needs the same tables:
      // in the cooperative launch each builds one slice of the entries,
      // publishes it and picks the rest up from L2 (building everything in
      // every block kept all SMs issue-bound for 4 us,
      // profiles/round2_timeline.md).
      {
        // (one piece per block: nobody waits for a slice its owner has not reached)
        const bool shared = a.shared_tables != nullptr && G.n_pieces > 1 && a.n_pieces <= (int)gridDim.x;
        const int n_all = G.n_fa + G.n_cm + G.n_rz;
        int e_lo = 0, e_hi = n_all;
        if (shared) {
          e_lo = (int)((int64_t)n_all * pi / G.n_pieces);
          e_hi = (int)((int64_t)n_all * (pi + 1) / G.n_pieces);
        }
        uint32_t *gt = shared ? a.shared_tables + (size_t)G.index * (2 * a.cap_fa + a.cap_cm + a.cap_rz)
                              : nullptr;
        QueryS Q{};
        const uint32_t *set0 = S.sq[0].set[0];
        const bool lq = lane < nq;
        if (lq) { Q = S.sq[lane].s; set0 = S.sq[lane].set[0]; }
        const bool is_acc = (Q.qflags & SKYOPT_Q_ACC) != 0;
        const bool ratio = Q.mem_op == SKYOPT_OP_RATIO;
#pragma unroll 1
        for (int i = e_lo + warp; i < e_hi; i += kFastWarps) {
          uint32_t m1, m2 = 0;
          if (i < G.n_fa) {
            const uint32_t key = S.d_fa[i];
            const double disk = S.d_disk[i];
            const uint32_t fl = key & 0xFFFFu, ak = key >> 16;
            const uint32_t akey = (ak == SKYOPT_NONE16) ? (uint32_t)(32 * SKYOPT_ACC_SET_WORDS) : ak;
            // flags / fixed-host group (the low 16 bits of the row key)
            bool ok = lq && ((fl ^ Q.val_lo) & Q.mask_lo & 0xFFFFu) == 0u;
            if (is_acc) ok = ok && ((set0[(akey >> 5) & 63u] >> (akey & 31u)) & 1u);
            if (Q.disk_op != 0)
              ok = ok && (Q.disk_op == SKYOPT_DISK_GE ? (disk >= Q.disk_size)
                                                      : (fabs(disk - Q.disk_size) < 1.0));
            m1 = __ballot_sync(0xFFFFFFFFu, ok);
            m2 = __ballot_sync(0xFFFFFFFFu, ok && ((fl & Q.flags2) == Q.flags2));
            if (lane == 0) {
              S.Tfa[i] = make_uint2(m1, m2);
              if (shared) { gt[2 * i] = m1; gt[2 * i + 1] = m2; }
            }
          } else if (i < G.n_fa + G.n_cm) {
            const int e = i - G.n_fa;
            const double2 v = S.d_cm[e];
            const double lo = ratio ? __dmul_rn(v.x, Q.mem_lo) : Q.mem_lo;
            const bool okc = (Q.cpus_op == 0) | ((v.x >= Q.cpu_lo) & (v.x <= Q.cpu_hi));
            const bool okr = (Q.mem_op == 0) | ((v.y >= lo) & (v.y <= Q.mem_hi));
            m1 = __ballot_sync(0xFFFFFFFFu, lq & okc & okr);
            if (lane == 0) { S.Tcm[e] = m1; if (shared) gt[2 * a.cap_fa + e] = m1; }
          } else {
            const int e = i - G.n_fa - G.n_cm;
            const uint32_t key = S.d_rz[e];  // region | zone << 16
            // region: row-key bits 16..31, zone: bits 32..47
            const bool ok = lq && (((key & 0xFFFFu) ^ (Q.val_lo >> 16)) & (Q.mask_lo >> 16)) == 0u &&
                            (((key >> 16) ^ Q.val_hi) & Q.mask_hi & 0xFFFFu) == 0u;
            m1 = __ballot_sync(0xFFFFFFFFu, ok);
            if (lane == 0) { S.Trz[e] = m1; if (shared) gt[2 * a.cap_fa + a.cap_cm + e] = m1; }
          }
        }
        if (shared) {
          // publish the slice, wait for the others, fetch the rest
          __syncthreads();
          if (tid == 0) {
            __threadfence();
            atomicAdd(a.group_ready + G.index, 1u);
            while (*reinterpret_cast<volatile unsigned int *>(a.group_ready + G.index) < (unsigned)G.n_pieces)
              if (!(a.noprune & 4u)) __nanosleep(32);
            __threadfence();
          }
          __syncthreads();
#pragma unroll 1
          for (int i = tid; i < n_all; i += kScanThreads) {
            if (i >= e_lo && i < e_hi) continue;
            if (i < G.n_fa) S.Tfa[i] = make_uint2(__ldcg(gt + 2 * i), __ldcg(gt + 2 * i + 1));
            else if (i < G.n_fa + G.n_cm) S.Tcm[i - G.n_fa] = __ldcg(gt + 2 * a.cap_fa + (i - G.n_fa));
            else S.Trz[i - G.n_fa - G.n_cm] = __ldcg(gt + 2 * a.cap_fa + a.cap_cm + (i - G.n_fa - G.n_cm));
          }
        }
      }
      __syncthreads();
      trace_mark(a.trace, 0, 2);
      if (tid == 0) trace_put(a.trace, 0, 7, (unsigned long long)(clock64() - c_tab));
    }
    // lane q <-> query q: what the zone-map test needs
    uint32_t req = 0, grp = 0, sg_lo = 0, sg_hi = 0;
    bool acc = false;
    if (lane < nq) {
      const QueryS &L = S.sq[lane].s;
      req = L.req_flags; grp = L.grp_bit; sg_lo = L.sig_lo; sg_hi = L.sig_hi;
      acc = (L.qflags & SKYOPT_Q_ACC) != 0;
    }
    uint32_t best = S.sbest[lane];
    uint32_t anyw = 0;

    auto test = [&](const uint4 &z, uint32_t cmn) -> uint32_t {
      if (!prune) return 0xFFFFFFFFu;
      const bool pass = lane < nq && ((z.x & req) == req) && ((z.w & grp) == grp) &&
                        (!acc || (((sg_lo & z.y) | (sg_hi & z.z)) != 0u)) && cmn < best;
      return __ballot_sync(0xFFFFFFFFu, pass);
    };

    // Software pipeline through a per-warp ring of kRingDepth chunk slots in
    // shared memory, filled with cp.async (no registers held by rows in
    // flight): the rows of chunks k+1 .. k+kRingDepth-1 are on their way
    // while chunk k is scored. The zone-map / bound test decides at issue
    // time whether a chunk is fetched at all.
    for (int j0 = 0; j0 < n_mine; j0 += 32) {
      const int nr = min(32, n_mine - j0);
      if (j0 > 0) {
        // next round of 32 chunks: summaries and the first fetch
        cp_wait<0>();
        __syncwarp();
        if (prune && lane < nr) {
          const int cl = chunk_begin + warp + kFastWarps * (j0 + lane);
          zs = ldg_nc_v4(a.cat.zone_map + cl);
          cms = ldg_nc_u32(a.f.cmin[col] + cl);
        }
        fetch_rows2(a, col, chunk_begin + warp + kFastWarps * j0, lane, ring[j0 % kRingDepth]);
        cp_commit();
      }
      // chunk j0 was fetched unconditionally; is it worth scoring?
      uint32_t live_bits = 0;
      auto live_of = [&](int k) -> bool {
        if (!prune) return true;
        uint4 z;
        z.x = __shfl_sync(0xFFFFFFFFu, zs.x, k); z.y = __shfl_sync(0xFFFFFFFFu, zs.y, k);
        z.z = __shfl_sync(0xFFFFFFFFu, zs.z, k); z.w = __shfl_sync(0xFFFFFFFFu, zs.w, k);
        const uint32_t c = __shfl_sync(0xFFFFFFFFu, cms, k);
        return test(z, c) != 0u;
      };
      if (live_of(0)) live_bits |= 1u;
      auto issue = [&](int k) {
        if (k < nr && live_of(k)) {
          fetch_rows2(a, col, chunk_begin + warp + kFastWarps * (j0 + k), lane, ring[(j0 + k) % kRingDepth]);
          live_bits |= 1u << k;
        }
        cp_commit();
      };
#pragma unroll
      for (int k = 1; k < kRingDepth - 1; ++k) issue(k);
#pragma unroll 1
      for (int k = 0; k < nr; ++k) {
        issue(k + kRingDepth - 1);
        cp_wait<kRingDepth - 1>();
        __syncwarp();
        if (a.trace) ++n_visit;
        if ((live_bits >> k) & 1u) {
          if (a.trace) ++n_live;
          const RingSlot &R = ring[(j0 + k) % kRingDepth];
          const uint4 rk = *reinterpret_cast<const uint4 *>(R.rk + 4 * lane);
          const uint2 cmv = *reinterpret_cast<const uint2 *>(R.cm + 4 * lane);
          const uint2 fav = *reinterpret_cast<const uint2 *>(R.fa + 4 * lane);
          const uint2 rzv = *reinterpret_cast<const uint2 *>(R.rz + 4 * lane);
          const uint32_t c0 = cmv.x & 0xFFFFu, c1 = cmv.x >> 16, c2 = cmv.y & 0xFFFFu, c3 = cmv.y >> 16;
          const uint32_t f0 = fav.x & 0xFFFFu, f1 = fav.x >> 16, f2 = fav.y & 0xFFFFu, f3 = fav.y >> 16;
          const uint32_t r0 = rzv.x & 0xFFFFu, r1 = rzv.x >> 16, r2 = rzv.y & 0xFFFFu, r3 = rzv.y >> 16;
          const uint2 a0 = S.Tfa[f0], a1 = S.Tfa[f1], a2 = S.Tfa[f2], a3 = S.Tfa[f3];
          const uint32_t z_0 = S.Trz[r0], z_1 = S.Trz[r1], z_2 = S.Trz[r2], z_3 = S.Trz[r3];
          const uint32_t m0 = a0.y & S.Tcm[c0] & z_0, m1 = a1.y & S.Tcm[c1] & z_1;
          const uint32_t m2 = a2.y & S.Tcm[c2] & z_2, m3 = a3.y & S.Tcm[c3] & z_3;
          // any_stage1 is only read for gate queries (GCP) and scan results
          if (G.need_any | a.force_any) anyw |= (a0.x & z_0) | (a1.x & z_1) | (a2.x & z_2) | (a3.x & z_3);
          const uint32_t many = m0 | m1 | m2 | m3;
          // lane q: which lanes hold a row query q accepts; lanes are in
          // ascending rank order, so the first one holds the chunk's argmin
          const uint32_t B = warp_transpose32(many, tl);
          const int src = B ? (__ffs(B) - 1) : 0;
          const uint32_t first = __shfl_sync(0xFFFFFFFFu, rk.x, src);
          const bool maybe = B != 0u && first < best;
          if (__any_sync(0xFFFFFFFFu, maybe)) {
            // which of that lane's four rows (ascending) is the first accepted
            const uint32_t q0 = __shfl_sync(0xFFFFFFFFu, m0, src), q1 = __shfl_sync(0xFFFFFFFFu, m1, src);
            const uint32_t q2 = __shfl_sync(0xFFFFFFFFu, m2, src);
            const uint32_t k1 = __shfl_sync(0xFFFFFFFFu, rk.y, src), k2 = __shfl_sync(0xFFFFFFFFu, rk.z, src);
            const uint32_t k3 = __shfl_sync(0xFFFFFFFFu, rk.w, src);
            if (maybe) {
              const uint32_t cand = ((q0 >> lane) & 1u) ? first : ((q1 >> lane) & 1u) ? k1
                                  : ((q2 >> lane) & 1u) ? k2 : k3;
              if (cand < best) best = cand;
            }
          }
        }
        __syncwarp();  // the slot is free before it is refilled
        if (prune && lane < nq) {
          // share the bound inside the block (any achieved rank is a valid bound)
          const uint32_t sb = S.sbest[lane];
          if (best < sb) atomicMin(&S.sbest[lane], best); else best = sb;
        }
      }
    }
    cp_wait<0>();
    // ---- publish: block minimum per query, any-match bits
    anyw = __reduce_or_sync(0xFFFFFFFFu, anyw);
    if (lane < nq && best != kRankNone) atomicMin(&S.sbest[lane], best);
    if (lane == 0 && anyw) atomicOr(&S.sany[0], anyw);
    __syncthreads();
    trace_mark(a.trace, 0, 3);
    if (tid < nq) {
      const int qid = S.sq[tid].qid;
      const uint32_t v = S.sbest[tid];
      if (v != kRankNone) atomicMin(a.best_rank + qid, v);
      if ((S.sany[0] >> tid) & 1u) atomicOr(a.any1 + qid, 1u);
    }
  }
  trace_mark(a.trace, 0, 4);
  if (a.trace && lane == 0 && blockIdx.x < kTraceBlocks) {
    atomicAdd(&a.trace[((size_t)blockIdx.x) * kTraceSlots + 5],
              (unsigned long long)n_visit | ((unsigned long long)n_live << 32));
  }
}

__global__ void __launch_bounds__(kScanThreads, 4) scan2_kernel(Scan2Args a) {
  extern __shared__ __align__(16) unsigned char smem2[];
  scan2_body(a, smem2);
}

// Scan results in the caller's shape (skyopt_scan / SkyoptSolution.scan).
__global__ void finalize2_kernel(CatDev cat, FastCat f, int n_queries,
                                 const SkyoptQuery *__restrict__ queries,
                                 const uint32_t *__restrict__ best_rank,
                                 const uint32_t *__restrict__ any_in,
                                 ScanFinal *__restrict__ finals, uint32_t *__restrict__ any1) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= n_queries) return;
  const SkyoptQuery Q = queries[q];
  ScanFinal out; out.key = kKeyNone; out.row = -1; out.inst = -1;
  const uint32_t r = best_rank[q];
  if (r != kRankNone) {
    const RankRec rec = f.rank_rec[Q.price_col ? 1 : 0][(int64_t)cat.cloud_row_offsets[Q.cloud] + r];
    if (rec.price <= Q.max_price) { out.key = price_key(rec.price); out.row = rec.row; out.inst = rec.inst; }
  }
  finals[q] = out;
  any1[q] = any_in[q];
}

// ---------------------------------------------------------------------------
// K2': block per task.

// What a task block needs of its task and DAG, in one record (host-prepared).
struct PlaceTask {
  int32_t slot_begin, slot_end;
  int32_t blocked_begin, blocked_end;
  int32_t minimize_cost;
  int32_t pad_[3];
};
static_assert(sizeof(PlaceTask) == 32, "PlaceTask layout");

// What a slot needs of its query (host-prepared): where the query's ranks
// decode and its price cap.
struct SlotAux {
  int64_t rec_base;     // cloud_row_offsets[query.cloud]
  int32_t qcol;         // the query's price column
  int32_t cloud_r0, cloud_r1;  // row range of the slot's cloud
  int16_t has_zones;
  int16_t acc_list_key;  // the one key of the slot's accelerator set, -1 = none
  double max_price;
};
static_assert(sizeof(SlotAux) == 32, "SlotAux layout");

// The cheapest candidate of one (task, cloud): what the chain DP needs of a
// task's candidate table. `idx` is the FIRST candidate (task order) with the
// smallest value; `v2` the smallest value among the cloud's candidates in front
// of it (all larger than vmin) -- the only ones that could take a first-minimum
// tie from it after rounding (skyopt_step.cuh, "hazard").
struct TaskMin {
  unsigned long long vmin;  // price_key(value), kKeyNone = the cloud has no candidate
  unsigned long long v2;    // price_key, kKeyNone = nothing in front
  int32_t idx;
  int32_t pad_[3];
};
static_assert(sizeof(TaskMin) == 32, "TaskMin layout");

struct PlaceArgs {
  CatDev cat;
  FastCat f;
  const PlaceTask *ptasks;
  const SlotAux *saux;
  const uint32_t *best_rank;
  const uint32_t *any1;
  const uint32_t *acc_sets;
  SolveIn in;
  SolveWork w;
  int32_t *task_n;
  TaskMin *task_mv;   // [n_tasks][n_clouds] cheapest candidate of every cloud, or null
  unsigned long long *trace;
};

struct PlaceSlot {
  int32_t inst;        // instance type expanded (-1: empty slot, -2: TPU-VM)
  int32_t host_off, host_n;  // host VM's static list (GCP accelerator slots)
  int32_t list_off, list_n;  // the list that is filtered into candidates
  int32_t kind;        // 0 empty, 1 instance list, 2 accelerator list
  int32_t cand_acc;
  int32_t n_e[2], n_b[2];  // kept before / after the blocked filter, [us, other]
  unsigned long long vmin; // price_key of the cheapest unblocked candidate's value
  unsigned long long v2;   // ... of the cheapest one in front of it (kKeyNone: none)
  int32_t vidx;            // first candidate (index in the task) with that value
  int2 res;                // reservation entries [x, y) of (cloud, inst); empty: none
};

struct PlaceSmem {
  double host[kFastWarps][kFastMaxZones];
  SkyoptSlot slot[kFastMaxTaskSlots];
  SlotAux aux[kFastMaxTaskSlots];
  PlaceSlot ps[kFastMaxTaskSlots];
  int base[kFastMaxTaskSlots + 1];
};

__device__ __forceinline__ void place_body(const PlaceArgs &a, int t, unsigned char *smem) {
  PlaceSmem &M = *reinterpret_cast<PlaceSmem *>(smem);
  PlaceSlot *ps = M.ps;
  SkyoptSlot *s_slot = M.slot;
  SlotAux *s_aux = M.aux;
  int *s_base = M.base;
  double (*s_host)[kFastMaxZones] = M.host;
  const CatDev &cat = a.cat;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  trace_mark(a.trace, 1, 0);
  const PlaceTask TK = a.ptasks[t];
  const int ns = TK.slot_end - TK.slot_begin;
  const double kNaN = __longlong_as_double(0x7FF8000000000000ll);

  // ---- phase A: what each slot expands (thread per slot)
  if (tid < ns) {
    const int s = TK.slot_begin + tid;
    const SkyoptSlot S = a.in.slots[s];
    const SlotAux X = a.saux[s];
    s_slot[tid] = S; s_aux[tid] = X;
    PlaceSlot p{};
    int inst = S.inst_id;
    bool empty = false;
    const int col = S.price_col ? 1 : 0;
    // independent loads first
    const uint32_t gate = (S.gate_query >= 0) ? __ldcg(a.any1 + S.gate_query) : 1u;
    const uint32_t r = (S.query >= 0) ? __ldcg(a.best_rank + S.query) : 0u;
    ListRec acc_rec{};
    if (S.acc_set >= 0 && X.acc_list_key >= 0) acc_rec = a.f.acc_list[X.acc_list_key];
    ListRec host{};
    if (gate == 0u) empty = true;
    if (S.query >= 0) {
      if (r == kRankNone) empty = true;
      else {
        const RankRec rec = a.f.rank_rec[X.qcol][X.rec_base + r];
        if (!(rec.price <= X.max_price)) empty = true;  // price cap (common.py:563, :681)
        inst = rec.inst;
        host.off = rec.list_off; host.cnt[0] = rec.cnt[0]; host.cnt[1] = rec.cnt[1]; host.acc_key = rec.acc_key;
        if (inst < 0) empty = true;
      }
    } else if (inst >= 0) {
      host = a.f.inst_list[inst];
    }
    if (empty || (inst < 0 && inst != -2)) {
      p.kind = 0; p.inst = -1;
    } else {
      p.inst = inst;
      int acc = S.cand_acc_key;
      if (acc < 0 && inst >= 0) acc = host.acc_key;
      p.cand_acc = acc;
      if (S.acc_set >= 0) {
        // the set holds exactly one key (checked on the host)
        p.kind = 2;
        p.list_off = acc_rec.off; p.list_n = acc_rec.cnt[col];
        if (inst >= 0) { p.host_off = host.off; p.host_n = host.cnt[col]; }
      } else {
        p.kind = 1;
        p.list_off = host.off;
        p.list_n = host.cnt[col];
      }
    }
    // the slot's reservation entries, searched once: lanes then look up
    // their candidate's zone inside this range only. Spot candidates and the
    // TIME objective never consume reserved nodes.
    p.res = make_int2(0, 0);
    if (a.in.n_res && TK.minimize_cost && !S.use_spot && p.kind != 0 && p.inst >= 0)
      p.res = reservation_range(a.in.res, a.in.n_res, S.cloud, p.inst);
    ps[tid] = p;
  }
  __syncthreads();
  trace_mark(a.trace, 1, 1);

  // One pass over a slot's static list by one warp.
  auto walk = [&](int ls, bool write, int base_e0, int base_e1, int base_b0, int base_b1) {
    PlaceSlot &p = ps[ls];
    const int s = TK.slot_begin + ls;
    const SkyoptSlot &S = s_slot[ls];
    const SlotAux &X = s_aux[ls];
    const int col = S.price_col ? 1 : 0;
    const bool has_zones = X.has_zones != 0;
    const bool split = S.split_by_zone && has_zones;
    const int reg0 = cat.cloud_region_offsets[S.cloud];
    const bool gcp = p.kind == 2;
    const ExpEnt *list = (gcp ? a.f.aexp_ent[col] : a.f.exp_ent[col]) + p.list_off;
    double *host = s_host[warp];
    if (gcp && p.inst >= 0) {
      // host VM price per zone (gcp.py:296-322)
#pragma unroll 1
      for (int i = lane; i < kFastMaxZones; i += 32) host[i] = kNaN;
      __syncwarp();
      const ExpEnt *hl = a.f.exp_ent[col] + p.host_off;
#pragma unroll 1
      for (int i = lane; i < p.host_n; i += 32) {
        const ExpEnt e = hl[i];
        if (e.zn != SKYOPT_NONE16 && e.zn < kFastMaxZones) host[e.zn] = e.price;
      }
      __syncwarp();
    }
    int ne0 = 0, ne1 = 0, nb0 = 0, nb1 = 0;
    unsigned long long vmin = kKeyNone;
    int vidx = 0x7FFFFFFF;
    const int64_t eoff = a.in.slot_off[s];
    const int64_t toff = a.in.task_off[t];
#pragma unroll 1
    for (int i0 = 0; i0 < p.list_n; i0 += 32) {
      const int i = i0 + lane;
      bool keep = i < p.list_n;
      ExpEnt e{};
      int rg = 0, zn = 0;
      double pa = 0.0, pb = 0.0;
      if (keep) {
        e = list[i];
        const int row = (int)(e.row & ~kRegionFirst);
        rg = e.rg; zn = e.zn;
        if (gcp && (row < X.cloud_r0 || row >= X.cloud_r1)) keep = false;
        if (S.region_id >= 0 && rg != S.region_id) keep = false;
        if (S.region_set >= 0 &&
            !test_bit(a.acc_sets + (int64_t)S.region_set * SKYOPT_ACC_SET_WORDS, (uint32_t)rg & 1023u))
          keep = false;  // image_id / ssh_proxy_command region allow-list
        if (S.zone_id >= 0 && (!has_zones || zn != S.zone_id)) keep = false;
        if (!split && S.zone_id < 0 && !(e.row & kRegionFirst)) keep = false;
        pa = e.price;
        if (gcp) {
          pb = pa;
          if (p.inst >= 0) {
            const double hb = (zn < kFastMaxZones) ? host[zn] : kNaN;
            if (hb != hb) keep = false;
            pa = hb;
          } else {
            pa = 0.0;
          }
        }
      }
      const bool other = keep && S.us_first && !cat.region_is_us[reg0 + rg];
      const int zout = (split || S.zone_id >= 0) ? (has_zones ? zn : -1) : -1;
      bool blocked = false;
      if (keep) {
#pragma unroll 1
        for (int b = TK.blocked_begin; b < TK.blocked_end; ++b) {
          const SkyoptBlocked Bk = a.in.blocked[b];
          const bool m = (Bk.cloud == -1 || Bk.cloud == S.cloud) &&
                         (Bk.inst_id == -1 || Bk.inst_id == p.inst) &&
                         (Bk.region_id == -1 || Bk.region_id == rg) &&
                         (Bk.zone_id == -1 || Bk.zone_id == zout) &&
                         (Bk.acc_key == -1 || Bk.acc_key == p.cand_acc) &&
                         (Bk.use_spot == -1 || Bk.use_spot == S.use_spot);
          if (m) { blocked = true; break; }
        }
      }
      const uint32_t ke0 = __ballot_sync(0xFFFFFFFFu, keep && !other);
      const uint32_t ke1 = __ballot_sync(0xFFFFFFFFu, keep && other);
      const uint32_t kb0 = __ballot_sync(0xFFFFFFFFu, keep && !other && !blocked);
      const uint32_t kb1 = __ballot_sync(0xFFFFFFFFu, keep && other && !blocked);
      if (write && keep) {
        const uint32_t below = (1u << lane) - 1u;
        const int pe = other ? base_e1 + ne1 + __popc(ke1 & below) : base_e0 + ne0 + __popc(ke0 & below);
        const int64_t ref = eoff + pe;
        a.in.ex.cand_region[ref] = rg;
        a.in.ex.cand_zone[ref] = zout;
        a.in.ex.cand_price_a[ref] = pa;
        a.in.ex.cand_price_b[ref] = pb;
        if (!blocked) {
          const int pbk = other ? base_b1 + nb1 + __popc(kb1 & below) : base_b0 + nb0 + __popc(kb0 & below);
          const int64_t o = toff + pbk;
          // float(hourly_cost * hours) * max(num_nodes - reserved, 0)
          const double hourly = __dadd_rn(pa, pb);
          a.w.tc_ref[o] = (int32_t)ref;
          a.w.tc_slot[o] = s;
          a.w.tc_cloud[o] = S.cloud;
          a.w.tc_hourly[o] = hourly;
          double mult = S.node_mult;
          if (p.res.y > p.res.x && zout >= 0) mult = reserved_node_mult(mult, reserved_in_range(a.in.res, p.res, zout));
          const double value = TK.minimize_cost ? __dmul_rn(__dmul_rn(hourly, S.hours), mult)
                                                : S.time_value;
          a.w.tc_value[o] = value;
          const unsigned long long vk = price_key(value);
          if (vk < vmin || (vk == vmin && pbk < vidx)) { vmin = vk; vidx = pbk; }
        }
      }
      ne0 += __popc(ke0); ne1 += __popc(ke1); nb0 += __popc(kb0); nb1 += __popc(kb1);
    }
    if (!write && lane == 0) { p.n_e[0] = ne0; p.n_e[1] = ne1; p.n_b[0] = nb0; p.n_b[1] = nb1; }
    if (write) {
      // cheapest value of the slot (the chain DP starts from per-cloud minima)
      const uint32_t hi = __reduce_min_sync(0xFFFFFFFFu, (uint32_t)(vmin >> 32));
      const uint32_t lo = __reduce_min_sync(0xFFFFFFFFu, ((uint32_t)(vmin >> 32) == hi) ? (uint32_t)vmin : 0xFFFFFFFFu);
      const unsigned long long vm = ((unsigned long long)hi << 32) | lo;
      const int first = (int)__reduce_min_sync(0xFFFFFFFFu, (vmin == vm) ? (uint32_t)vidx : 0x7FFFFFFFu);
      // candidates of the slot in front of the first minimum (none when the
      // list is in price order, the usual case)
      unsigned long long v2 = kKeyNone;
      if (vm != kKeyNone && first > base_b0) {
        __syncwarp();
#pragma unroll 1
        for (int j = base_b0 + lane; j < first; j += 32) {
          const unsigned long long k = price_key(__ldcg(a.w.tc_value + toff + j));
          if (k < v2) v2 = k;
        }
        const uint32_t h2 = __reduce_min_sync(0xFFFFFFFFu, (uint32_t)(v2 >> 32));
        const uint32_t l2 = __reduce_min_sync(0xFFFFFFFFu, ((uint32_t)(v2 >> 32) == h2) ? (uint32_t)v2 : 0xFFFFFFFFu);
        v2 = ((unsigned long long)h2 << 32) | l2;
      }
      if (lane == 0) { p.vmin = vm; p.vidx = first; p.v2 = v2; }
    }
  };

  // ---- phase B: count, then write (one copy of the walk: this code runs
  // once per launch, its size is its cost)
#pragma unroll 1
  for (int pass = 0; pass < 2; ++pass) {
    const bool write = pass == 1;
#pragma unroll 1
    for (int ls = warp; ls < ns; ls += kFastWarps) {
      if (ps[ls].kind != 0)
        walk(ls, write, 0, write ? ps[ls].n_e[0] : 0, write ? s_base[ls] : 0,
             write ? s_base[ls] + ps[ls].n_b[0] : 0);
      else if (lane == 0) { ps[ls].n_e[0] = ps[ls].n_e[1] = ps[ls].n_b[0] = ps[ls].n_b[1] = 0; ps[ls].vmin = kKeyNone; }
    }
    if (write) break;
    __syncthreads();
    trace_mark(a.trace, 1, 2);
    if (tid == 0) {
      int acc = 0;
#pragma unroll 1
      for (int i = 0; i < ns; ++i) { s_base[i] = acc; acc += ps[i].n_b[0] + ps[i].n_b[1]; }
      s_base[ns] = acc;
      a.task_n[t] = acc;
    }
    if (tid < ns) {
      const int s = TK.slot_begin + tid;
      a.in.ex.slot_count[s] = ps[tid].n_e[0] + ps[tid].n_e[1];
      a.in.ex.slot_inst[s] = ps[tid].inst;
    }
    __syncthreads();
  }
  if (a.task_mv) {
    __syncthreads();
    if (tid < cat.n_clouds) {
      // slots are in candidate order: a later slot only wins with a strictly
      // smaller value, and then everything seen so far is in front of it
      TaskMin m; m.vmin = kKeyNone; m.v2 = kKeyNone; m.idx = 0x7FFFFFFF; m.pad_[0] = m.pad_[1] = m.pad_[2] = 0;
#pragma unroll 1
      for (int i = 0; i < ns; ++i) {
        if (s_slot[i].cloud != tid || ps[i].kind == 0 || ps[i].vmin == kKeyNone) continue;
        if (ps[i].vmin < m.vmin) {
          m.v2 = m.vmin < ps[i].v2 ? m.vmin : ps[i].v2;
          m.vmin = ps[i].vmin; m.idx = ps[i].vidx;
        }
      }
      a.task_mv[(int64_t)t * cat.n_clouds + tid] = m;
    }
  }
  trace_mark(a.trace, 1, 3);
}

__global__ void __launch_bounds__(kScanThreads) place_kernel(PlaceArgs a) {
  extern __shared__ __align__(16) unsigned char smem_place[];
  place_body(a, blockIdx.x, smem_place);
}

}  // namespace skyopt
