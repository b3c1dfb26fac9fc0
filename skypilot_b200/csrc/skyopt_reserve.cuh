// Capacity reservations on the device: how many reserved nodes a launchable
// (cloud, instance type, zone) may consume, looked up in the problem's
// SkyoptReservation table (sorted by (cloud, inst_id, zone_id), unique).
// The reference prices such a candidate at
//   cost_per_node * max(num_nodes - reserved, 0)   (sky/optimizer.py:344-354)
// so reserved capacity costs nothing. Used by place_body (skyopt_fast.cuh)
// and gather_kernel (skyopt_kernels.cuh).
#pragma once

#include <stdint.h>

#include "skyopt.h"

namespace skyopt {

// Entries [x, y) of (cloud, inst) in the table: two lower-bound searches.
__device__ __forceinline__ int2 reservation_range(const SkyoptReservation *__restrict__ res, int n,
                                                  int cloud, int inst) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    const int c = __ldg(&res[mid].cloud), i = __ldg(&res[mid].inst_id);
    if (c < cloud || (c == cloud && i < inst)) lo = mid + 1; else hi = mid;
  }
  const int begin = lo;
  hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    const int c = __ldg(&res[mid].cloud), i = __ldg(&res[mid].inst_id);
    if (c < cloud || (c == cloud && i <= inst)) lo = mid + 1; else hi = mid;
  }
  return make_int2(begin, lo);
}

// Reserved nodes of `zone` among the entries [range.x, range.y) of one
// (cloud, instance type); 0 when the zone has none.
__device__ __forceinline__ int reserved_in_range(const SkyoptReservation *__restrict__ res, int2 range,
                                                 int zone) {
  int lo = range.x, hi = range.y;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(&res[mid].zone_id) < zone) lo = mid + 1; else hi = mid;
  }
  return (lo < range.y && __ldg(&res[lo].zone_id) == zone) ? __ldg(&res[lo].available) : 0;
}

// Reserved nodes of one launchable (cloud, instance type, zone).
__device__ __forceinline__ int reserved_nodes(const SkyoptReservation *__restrict__ res, int n,
                                              int cloud, int inst, int zone) {
  return reserved_in_range(res, reservation_range(res, n, cloud, inst), zone);
}

// max(num_nodes - reserved, 0): exact, node_mult is the integer num_nodes.
// Without reserved nodes it is node_mult itself, so the value
// hourly * hours * node_mult is bit-identical to a problem without a table.
__device__ __forceinline__ double reserved_node_mult(double node_mult, int reserved) {
  return reserved > 0 ? fmax(__dsub_rn(node_mult, (double)reserved), 0.0) : node_mult;
}

}  // namespace skyopt
