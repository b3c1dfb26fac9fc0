"""Capacity reservations: reserved nodes cost nothing in the COST objective.

A user who holds reserved capacity tells SkyPilot to use it in the config:

    aws:
      prioritize_reservations: true
      specific_reservations: [cr-0123456789abcdef0]
    gcp:
      specific_reservations: [projects/p/reservations/a100-pool]

The reference then prices a launchable at
`cost_per_node * max(num_nodes - reserved, 0)` (sky/optimizer.py:259-354),
where `reserved` is the number of reserved nodes the launchable may consume
in its zone, and AWS lists on-demand candidates per zone
(`AWS.optimize_by_zone`, sky/clouds/aws.py:369-371).

Like the enabled clouds (check.py), the reservations themselves are injected,
never fetched from a cloud API here:

  * `set_reservations([...])` -- a snapshot of `Reservation` records (tests,
    offline use, benchmarks), or None to clear it;
  * `set_reservations_provider(fn)` -- `fn(cloud_name)` returns that cloud's
    active reservations as `Reservation` records; it is called at most once per
    cloud whose config enables reservations, for each optimize call, batch or
    session open. INTEGRATION.md shows a binding to
    `describe_capacity_reservations` and `gcloud compute reservations list`.

The gating and consumability rule lives in `_rule` only: it answers
`Resources.get_reservations_available_resources()` and builds the device
table (`device_table`) that the kernels look every candidate up in.
"""
import dataclasses
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import numpy as np

from skypilot_b200 import _native
from skypilot_b200 import skypilot_config

# clouds whose reservations the reference reads (aws.py:1490-1519,
# gcp.py:1419-1438); every other cloud counts 0 (cloud.py:512-525)
RESERVATION_CLOUDS = ('aws', 'gcp')


@dataclasses.dataclass(frozen=True)
class Reservation:
    """One active reservation.

    cloud          registered cloud name ('aws', 'gcp', ...)
    name           AWS: CapacityReservationId; GCP: projects/<p>/reservations/<r>
    instance_type  AWS: InstanceType; GCP: the machine type (the host VM of a
                   GPU candidate, e.g. n1-highmem-8)
    region, zone   where the capacity is
    available      consumable nodes (AWS AvailableInstanceCount; GCP
                   specificReservation.count - inUseCount)
    targeted       AWS InstanceMatchCriteria == 'targeted'; GCP
                   specificReservationRequired: only usable when `name` is
                   listed in `<cloud>.specific_reservations`
    """
    cloud: str
    name: str
    instance_type: str
    region: str
    zone: str
    available: int
    targeted: bool = False


_records: Optional[Tuple[Reservation, ...]] = None
_provider: Optional[Callable[[str], Sequence[Reservation]]] = None
_generation = 0


def generation() -> int:
    """Bumped by every set_reservations / set_reservations_provider."""
    return _generation


def _changed() -> None:
    global _generation
    _generation += 1


def _validate(records: Sequence[Reservation]) -> Tuple[Reservation, ...]:
    from skypilot_b200.utils import registry  # pylint: disable=import-outside-toplevel
    out = []
    seen = set()
    for r in records:
        if not isinstance(r, Reservation):
            raise ValueError(f'not a Reservation: {r!r}')
        cloud = str(r.cloud).lower()
        if cloud not in registry.CLOUD_REGISTRY:
            raise ValueError(f'reservation {r.name!r}: unknown cloud '
                             f'{r.cloud!r}')
        if not r.zone:
            raise ValueError(f'reservation {r.name!r}: no zone')
        if (isinstance(r.available, bool) or
                not isinstance(r.available, (int, np.integer))):
            raise ValueError(f'reservation {r.name!r}: available must be an '
                             f'integer, got {r.available!r}')
        if r.available < 0:
            raise ValueError(f'reservation {r.name!r}: negative available '
                             f'count {r.available}')
        key = (cloud, r.name, r.zone)
        if key in seen:
            raise ValueError(f'reservation {r.name!r} listed twice in zone '
                             f'{r.zone!r}')
        seen.add(key)
        out.append(dataclasses.replace(r, cloud=cloud,
                                       available=int(r.available),
                                       targeted=bool(r.targeted)))
    return tuple(out)


def set_reservations(records: Optional[Sequence[Reservation]]) -> None:
    """Installs a snapshot of active reservations (None: no snapshot)."""
    global _records
    _records = None if records is None else _validate(list(records))
    _changed()


def set_reservations_provider(
        provider: Optional[Callable[[str], Sequence[Reservation]]]) -> None:
    """`provider(cloud_name)` -> that cloud's active reservations. A snapshot
    installed with set_reservations takes precedence."""
    global _provider
    _provider = provider
    _changed()


def need_to_query_reservations() -> bool:
    """sky/utils/resources_utils.py:425-451: some cloud's config sets
    `specific_reservations` or a truthy `prioritize_reservations`."""
    from skypilot_b200.utils import registry  # pylint: disable=import-outside-toplevel
    for cloud in registry.CLOUD_REGISTRY.keys():
        if (skypilot_config.get_effective_region_config(
                cloud, None, ('specific_reservations',), None) is not None or
                skypilot_config.get_effective_region_config(
                    cloud, None, ('prioritize_reservations',), False)):
            return True
    return False


def use_reservations(cloud: str) -> bool:
    """Whether `cloud` consults its reservations at all: AWS
    `aws_utils.use_reservations()` (clouds/utils/aws_utils.py:30-41), GCP
    `_list_reservations_for_instance_type` (clouds/utils/gcp_utils.py:142-152).
    Both: a truthy prioritize_reservations or a non-empty
    specific_reservations."""
    if cloud not in RESERVATION_CLOUDS:
        return False
    return bool(
        skypilot_config.get_effective_region_config(
            cloud, None, ('prioritize_reservations',), False) or
        skypilot_config.get_effective_region_config(
            cloud, None, ('specific_reservations',), None))


def _specific(cloud: str) -> set:
    names = skypilot_config.get_effective_region_config(
        cloud, None, ('specific_reservations',), None)
    return set(names or ())


def _rule(cloud: str) -> Optional[Callable[[Reservation], bool]]:
    """The one gating + consumability rule. None: the cloud's reservations
    are not consulted (every candidate counts 0). Otherwise a predicate: a
    reservation counts if it is not targeted, or if its name is listed in
    `<cloud>.specific_reservations` (AWS aws.py:1506-1512, GCP
    gcp_utils.py:94-103)."""
    if not use_reservations(cloud):
        return None
    specific = _specific(cloud)
    return lambda r: not r.targeted or r.name in specific


def _cloud_records(cloud: str) -> List[Reservation]:
    """Active reservations of one cloud: the snapshot, else the provider."""
    if _records is not None:
        return [r for r in _records if r.cloud == cloud]
    if _provider is None:
        return []
    return [r for r in _validate(list(_provider(cloud) or ()))
            if r.cloud == cloud]


def _zone_matches(cloud: str, record: Reservation, region: str,
                  zone: str) -> bool:
    if cloud == 'aws':
        # listed per (instance type, region), matched by zone name
        return record.region == region and record.zone == zone
    # GCP lists per machine type and matches the zone only
    return record.zone == zone


def available_resources(cloud: str, instance_type: str, region: str,
                        zone: Optional[str],
                        use_spot: bool) -> Dict[str, int]:
    """{reservation name: consumable nodes} of one launchable: the result of
    Resources.get_reservations_available_resources (sky/resources.py:
    1785-1812)."""
    cloud = cloud.lower()
    if use_spot or cloud not in RESERVATION_CLOUDS:
        return {}
    if zone is None:
        # aws.py:1498-1501, gcp.py:1427-1431
        return {name: 0 for name in _specific(cloud)}
    rule = _rule(cloud)
    if rule is None:
        return {}
    return {
        r.name: r.available
        for r in _cloud_records(cloud)
        if r.instance_type == instance_type and
        _zone_matches(cloud, r, region, zone) and rule(r)
    }


_EMPTY = np.zeros(1, dtype=_native.RESERVATION_DTYPE)


def device_table(store) -> Tuple[np.ndarray, int]:
    """(SkyoptReservation array, number of entries) for `store`: consumable
    reserved nodes summed per (cloud, instance type id, zone id), sorted and
    unique. Records of instance types or zones the catalog does not have
    count 0, like in the reference. Without a reservation config the table
    is empty and the device takes no look-up.

    A snapshot's table is memoised per (store, snapshot, config); a provider
    is asked again on every call."""
    if not need_to_query_reservations():
        return _EMPTY, 0
    key = (_generation, skypilot_config.generation())
    if _records is not None:
        hit = store.__dict__.get('_reservation_table')
        if hit is not None and hit[0] == key:
            return hit[1], hit[2]
    sums: Dict[Tuple[int, int, int], int] = {}
    for cloud in RESERVATION_CLOUDS:
        rule = _rule(cloud)
        if rule is None or not store.has_cloud(cloud):
            continue
        table = store.cloud(cloud)
        for r in _cloud_records(cloud):
            if r.available <= 0 or not rule(r):
                continue
            inst = table.inst_index.get(r.instance_type)
            zone = table.zone_exact.get(r.zone)
            if inst is None or zone is None:
                continue
            if cloud == 'aws':
                region = table.region_exact.get(r.region)
                if region is None or table.zone_region[zone] != region:
                    continue
            k = (table.index, inst, zone)
            sums[k] = sums.get(k, 0) + r.available
    if not sums:
        arr, n = _EMPTY, 0
    else:
        keys = sorted(sums)
        arr = np.zeros(len(keys), dtype=_native.RESERVATION_DTYPE)
        arr['cloud'] = [k[0] for k in keys]
        arr['inst_id'] = [k[1] for k in keys]
        arr['zone_id'] = [k[2] for k in keys]
        arr['available'] = [min(sums[k], 0x7FFFFFFF) for k in keys]
        n = len(keys)
    if _records is not None:
        store.__dict__['_reservation_table'] = (key, arr, n)
    return arr, n
