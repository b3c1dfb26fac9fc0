"""Host-side assembly of libskyopt problems and the calls into the device.

A `ProblemBuilder` collects catalog queries (constraint vectors), expansion
slots, tasks and DAGs as numpy structured arrays (layouts of include/skyopt.h)
and hands them to `skyopt_optimize` / `skyopt_scan` in ONE call; all row-level
work (filter, argmin, region/zone expansion, cost, blocked filter, DP) happens
on the GPU. There is no CPU implementation behind these calls.
"""
import ctypes
import math
import struct
import functools
import operator
import re
from typing import Any, Dict, List, Optional, Sequence, Tuple

import numpy as np

from skypilot_b200.utils import timeline
from skypilot_b200 import _native
from skypilot_b200.catalog.store import CatalogStore
from skypilot_b200.utils import resources_utils

NO_MATCH_ID = 65534  # a region / zone id no row carries
_INF = float('inf')


def _addr(arr: np.ndarray) -> int:
    """Address of a numpy buffer. (`__array_interface__` is no shortcut: for
    a structured dtype it rebuilds the field description on every access.)"""
    return arr.ctypes.data


@functools.lru_cache(maxsize=4096)
def parse_cpus(cpus: Optional[str]) -> Tuple[int, float]:
    """'8' -> (EQ, 8.0), '8+' -> (GE, 8.0) (sky/catalog/common.py:431-452)."""
    if cpus is None:
        return _native.OP_NONE, 0.0
    text = str(cpus)
    body = text[:-1] if text.endswith('+') else text
    try:
        value = float(body)
    except ValueError:
        raise ValueError('The "cpus" field should be either a number or '
                         f'a string "<number>+". Found: {cpus!r}') from None
    return (_native.OP_GE if text.endswith('+') else _native.OP_EQ), value


@functools.lru_cache(maxsize=4096)
def parse_memory(memory: Optional[str]) -> Tuple[int, float]:
    """'16' EQ, '16+' GE, '4x' RATIO (sky/catalog/common.py:455-478)."""
    if memory is None:
        return _native.OP_NONE, 0.0
    text = str(memory)
    body = text[:-1] if text.endswith(('+', 'x')) else text
    try:
        value = float(body)
    except ValueError:
        raise ValueError(
            'The "memory" field should be either a number or a string '
            f'"<number>+" or "<number>x". Found: {memory!r}') from None
    if text.endswith('+'):
        return _native.OP_GE, value
    if text.endswith('x'):
        return _native.OP_RATIO, value
    return _native.OP_EQ, value


def region_filter_id(table, region: Optional[str]) -> int:
    """Case-insensitive region filter of _filter_region_zone (common.py:509)."""
    if region is None:
        return -1
    return table.region_lower.get(region.lower(), NO_MATCH_ID)


def zone_filter_id(table, zone: Optional[str]) -> int:
    if zone is None:
        return -1
    return table.zone_lower.get(zone.lower(), NO_MATCH_ID)


def region_exact_id(table, region: Optional[str]) -> int:
    """Exact-name filter of regions_with_offering (aws.py:360-367)."""
    if region is None:
        return -1
    return table.region_exact.get(region, NO_MATCH_ID)


def zone_exact_id(table, zone: Optional[str]) -> int:
    if zone is None:
        return -1
    return table.zone_exact.get(zone, NO_MATCH_ID)


_PLAIN_NAME = re.compile(r'[A-Za-z0-9_\- ]+')


def accelerator_sets(store: CatalogStore, acc_name: str,
                     acc_count) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Dictionary-level accelerator predicates -> key bitmasks.

    exact   name.fullmatch(acc, case=False) & |count - c| <= 0.01
            (common.py:657-658)
    fuzzy   name.contains(acc, case=False)  & count >= c   (common.py:661-663)
    strict  name.fullmatch(acc, case=False) & count == c   (GCP
            _get_accelerator, gcp_catalog.py:404-417)
    The string predicates run once per distinct (name, count) pair of the
    catalog dictionary; rows carry only the pair's id.
    """
    cache = store.__dict__.setdefault('_acc_set_cache', {})
    hit = cache.get((acc_name, float(acc_count)))
    if hit is not None:
        return hit
    count = float(acc_count)
    if _PLAIN_NAME.fullmatch(acc_name):
        # A name without regex metacharacters: case-insensitive fullmatch is
        # equality of the lower-cased names, `contains` a substring test --
        # answered from the store's name index (a property of the catalog
        # dictionary, not a request memo) instead of a regex per key.
        index = store.__dict__.get('_acc_name_index')
        if index is None:
            index = {}
            for k, (name, cnt) in enumerate(store.acc_keys):
                index.setdefault(name.lower(), []).append((k, cnt))
            store.__dict__['_acc_name_index'] = index
        low = acc_name.lower()
        # bitmasks as Python ints (one shift-or per key), turned into the
        # uint32 words of the C ABI once
        e_bits = f_bits = s_bits = 0
        for name, keys in index.items():
            if low not in name:
                continue
            same = name == low
            for k, cnt in keys:
                if cnt >= count:
                    f_bits |= 1 << k
                if same:
                    if abs(cnt - count) <= 0.01:
                        e_bits |= 1 << k
                    if cnt == count:
                        s_bits |= 1 << k
        nbytes = 4 * _native.ACC_SET_WORDS
        exact, fuzzy, strict = (np.frombuffer(
            bits.to_bytes(nbytes, 'little'), dtype=np.uint32)
                                for bits in (e_bits, f_bits, s_bits))
        cache[(acc_name, float(acc_count))] = (exact, fuzzy, strict)
        return exact, fuzzy, strict
    pattern = re.compile(acc_name, flags=re.IGNORECASE)
    exact = store.accelerator_set(lambda n, c: pattern.fullmatch(n) is not None
                                  and abs(c - count) <= 0.01)
    fuzzy = store.accelerator_set(
        lambda n, c: pattern.search(n) is not None and c >= count)
    strict = store.accelerator_set(lambda n, c: pattern.fullmatch(n) is not None
                                   and c == count)
    # The dictionary is immutable once the store is built, so the three
    # bitmasks are a pure function of (name, count).
    cache[(acc_name, float(acc_count))] = (exact, fuzzy, strict)
    return exact, fuzzy, strict


def format_fuzzy(store: CatalogStore, keys: Sequence[int]) -> List[str]:
    """'A100:8' / 'A10:0.17' strings (sky/catalog/common.py:668-675)."""
    out = []
    for k in keys:
        name, count = store.acc_keys[int(k)]
        shown = int(count) if float(count).is_integer() else f'{count:.2f}'
        out.append(f'{name}:{shown}')
    return out


def set_id(store: CatalogStore, key: bytes) -> int:
    """Store-wide id of an accelerator-key bitmask (registered on first use;
    the table is tiny: a few dozen 128-byte sets per catalog)."""
    reg = store.__dict__.setdefault('_set_registry', {})
    idx = reg.get(key)
    if idx is None:
        idx = len(reg)
        reg[key] = idx
        store.__dict__.pop('_set_table', None)
    return idx


def set_table(store: CatalogStore) -> np.ndarray:
    table = store.__dict__.get('_set_table')
    if table is None:
        reg = store.__dict__.get('_set_registry', {})
        table = np.frombuffer(b''.join(reg.keys()), dtype=np.uint32).copy() if (
            reg) else np.zeros(0, dtype=np.uint32)
        store.__dict__['_set_table'] = table
    return table


_MINUS_ONE_DEFAULT = frozenset(('acc_set', 'fuzzy_set', 'region_id',
                                'zone_id', 'region_set'))
_PACKERS: Dict[Any, Tuple[struct.Struct, Tuple[str, ...]]] = {}
_FORMATS = {'i4': 'i', 'u4': 'I', 'f8': 'd', 'i8': 'q', 'u8': 'Q', 'u2': 'H',
            'i2': 'h'}


def _packer(dtype: np.dtype) -> Tuple[struct.Struct, Tuple[str, ...]]:
    """struct.Struct equivalent of an aligned numpy record dtype."""
    key = id(dtype)
    hit = _PACKERS.get(key)
    if hit is not None:
        return hit
    fmt, names, offset = '<', [], 0
    for name in dtype.names:
        field_dtype, field_offset = dtype.fields[name][:2]
        if field_offset > offset:
            fmt += f'{field_offset - offset}x'
        code = _FORMATS[field_dtype.str.lstrip('<=|')]
        if name == 'pad_':
            fmt += f'{field_dtype.itemsize}x'
        else:
            fmt += code
            names.append(name)
        offset = field_offset + field_dtype.itemsize
    if dtype.itemsize > offset:
        fmt += f'{dtype.itemsize - offset}x'
    packer = struct.Struct(fmt)
    assert packer.size == dtype.itemsize, (packer.size, dtype.itemsize)
    _PACKERS[key] = (packer, tuple(names))
    return _PACKERS[key]


def _defaults(dtype: np.dtype, overrides: Dict[str, Any]) -> Dict[str, Any]:
    base = {n: (-1 if n in _MINUS_ONE_DEFAULT else 0) for n in dtype.names
            if n != 'pad_'}
    base.update(overrides)
    return base


# every field of a record with its default; itemgetter pulls them out in
# struct order at C speed
_QUERY_DEFAULTS = _defaults(_native.QUERY_DTYPE, {})
_SLOT_DEFAULTS = _defaults(_native.SLOT_DTYPE, {
    'query': -1, 'inst_id': -1, 'gate_query': -1, 'cand_acc_key': -1,
    'hours': 1.0, 'node_mult': 1.0, 'time_value': 3600.0})
_DEFAULT_COST = (1.0, 1.0, 3600.0)
_QUERY_PACK = _packer(_native.QUERY_DTYPE)[0].pack
_QUERY_FIELDS = operator.itemgetter(*_packer(_native.QUERY_DTYPE)[1])
_SLOT_PACK = _packer(_native.SLOT_DTYPE)[0].pack
_SLOT_FIELDS = operator.itemgetter(*_packer(_native.SLOT_DTYPE)[1])
_TASK_PACK = _packer(_native.TASK_DTYPE)[0].pack
_TASK_FIELDS = operator.itemgetter(*_packer(_native.TASK_DTYPE)[1])


class ProblemBuilder:
    """Accumulates one batch for the device.

    Queries and slots are kept as packed records (bytes of the C structs), so
    that replaying a cached plan (Cloud.plan_cached) is a list append and
    `pack()` is one `b''.join` per table instead of a Python loop per field.
    Accelerator-key sets are registered once per catalog store and referenced
    by a store-wide id.
    """

    def __init__(self, store: CatalogStore):
        self.store = store
        self.query_recs: List[bytes] = []
        self.slot_recs: List[bytes] = []
        self.slot_qbase: List[int] = []
        # (hours, node_mult, time_value) of every slot, flat: three floats
        # per slot, patched into the records by one numpy pass in pack()
        self.slot_cost: List[float] = []
        self.task_recs: List[bytes] = []
        self.tasks: List[Dict[str, Any]] = []
        self.parents: List[int] = []
        self.tariffs: List[float] = []
        self.blocked: List[Dict[str, int]] = []
        self.dags: List[Dict[str, int]] = []
        # reserved capacity (reservations.device_table): one table for every
        # DAG of the batch; None = not stated yet, treated as empty
        self.reservations: Optional[Tuple[np.ndarray, int]] = None

    @property
    def n_queries(self) -> int:
        return len(self.query_recs)

    @property
    def n_slots(self) -> int:
        return len(self.slot_recs)

    # -- sets / queries -----------------------------------------------------
    def add_set(self, words: Optional[np.ndarray]) -> int:
        if words is None:
            return -1
        # the bitmask arrays of accelerator_sets() live as long as the store's
        # memo: their ids are remembered by object
        by_obj = self.store.__dict__.setdefault('_set_id_by_obj', {})
        hit = by_obj.get(id(words))
        if hit is not None and hit[0] is words:
            return hit[1]
        idx = set_id(self.store,
                     np.ascontiguousarray(words, dtype=np.uint32).tobytes())
        if len(by_obj) < 4096:
            by_obj[id(words)] = (words, idx)
        return idx

    @staticmethod
    def _record(fields: Dict[str, Any], dtype: np.dtype) -> bytes:
        """One C struct as bytes (struct.pack with the dtype's exact layout:
        an order of magnitude cheaper than a one-element numpy record)."""
        packer, names = _packer(dtype)
        get = fields.get
        return packer.pack(*[
            get(n, -1 if n in _MINUS_ONE_DEFAULT else 0) for n in names
        ])

    def replay_query(self, recorder: 'ProblemBuilder', i: int) -> int:
        """Copies query `i` of a recorded plan (Cloud.plan_cached)."""
        self.query_recs.append(recorder.query_recs[i])
        return len(self.query_recs) - 1

    def replay_slot(self, recorder: 'ProblemBuilder', i: int,
                    qbase: int) -> int:
        """Copies slot `i` of a recorded plan whose queries were replayed
        starting at index `qbase`."""
        self.slot_recs.append(recorder.slot_recs[i])
        self.slot_qbase.append(qbase)
        self.slot_cost.extend(_DEFAULT_COST)
        return len(self.slot_recs) - 1

    def set_slot_cost(self, slot: int, hours: float, node_mult: float,
                      time_value: float) -> None:
        self.slot_cost[3 * slot:3 * slot + 3] = (hours, node_mult, time_value)

    def add_query(self, spec: Dict[str, Any]) -> int:
        q = dict(_QUERY_DEFAULTS)
        q.update(spec)
        q['acc_set'] = self.add_set(q.pop('acc_words', None))
        q['fuzzy_set'] = self.add_set(q.pop('fuzzy_words', None))
        self.query_recs.append(_QUERY_PACK(*_QUERY_FIELDS(q)))
        return len(self.query_recs) - 1

    def cpus_mem_query(self,
                       cloud: str,
                       cpus: Optional[str],
                       memory: Optional[str],
                       region: Optional[str] = None,
                       zone: Optional[str] = None,
                       use_spot: bool = False,
                       max_hourly_cost: Optional[float] = None,
                       *,
                       flags_require: int = 0,
                       group: int = 0,
                       local_disk: Optional[str] = None) -> Dict[str, Any]:
        """Constraint vector of get_instance_type_for_cpus_mem_impl
        (sky/catalog/common.py:518-569)."""
        table = self.store.cloud(cloud) if isinstance(cloud, str) else cloud
        cop, cval = parse_cpus(cpus)
        mop, mval = parse_memory(memory)
        # Spot prices only order the rows when a price cap is set
        # (common.py:557-561).
        spot = bool(use_spot and max_hourly_cost is not None)
        spec = {
            'cloud': table.index, 'qflags': 0,
            'flags_require': flags_require | _native.F_HAS_INSTANCE,
            'group': group, 'price_col': 1 if spot else 0,
            'cpus_op': cop, 'cpus': cval, 'mem_op': mop, 'mem': mval,
            'region_id': region_filter_id(table, region),
            'zone_id': zone_filter_id(table, zone),
            'max_price': _INF if max_hourly_cost is None else float(
                max_hourly_cost),
        }
        _apply_local_disk(spec, local_disk)
        return spec

    def accelerator_query(self,
                          cloud: str,
                          acc_name: str,
                          acc_count,
                          cpus: Optional[str] = None,
                          memory: Optional[str] = None,
                          use_spot: bool = False,
                          region: Optional[str] = None,
                          zone: Optional[str] = None,
                          max_hourly_cost: Optional[float] = None,
                          *,
                          local_disk: Optional[str] = None,
                          flags_require2: int = 0,
                          want_list: bool = False,
                          want_fuzzy: bool = True) -> Dict[str, Any]:
        """Constraint vector of get_instance_type_for_accelerator_impl
        (sky/catalog/common.py:641-694)."""
        table = self.store.cloud(cloud) if isinstance(cloud, str) else cloud
        exact, fuzzy, _ = accelerator_sets(self.store, acc_name, acc_count)
        cop, cval = parse_cpus(cpus)
        mop, mval = parse_memory(memory)
        qflags = _native.Q_ACC
        if want_fuzzy:
            qflags |= _native.Q_FUZZY
        if want_list:
            qflags |= _native.Q_LIST
            if max_hourly_cost is None:
                qflags |= _native.Q_KEEP_NAN
        spec = {
            'cloud': table.index, 'qflags': qflags, 'flags_require': 0,
            'flags_require2': flags_require2,
            'acc_words': exact, 'fuzzy_words': fuzzy if want_fuzzy else None,
            'price_col': 1 if use_spot else 0,
            'cpus_op': cop, 'cpus': cval, 'mem_op': mop, 'mem': mval,
            'region_id': region_filter_id(table, region),
            'zone_id': zone_filter_id(table, zone),
            'max_price': _INF if max_hourly_cost is None else float(
                max_hourly_cost),
        }
        _apply_local_disk(spec, local_disk)
        return spec

    # -- slots / tasks / dags ----------------------------------------------
    def add_slot(self, **fields) -> int:
        slot = dict(_SLOT_DEFAULTS)
        words = fields.pop('acc_words', None)
        region_words = fields.pop('region_words', None)
        slot.update(fields)
        if words is not None:
            slot['acc_set'] = self.add_set(words)
        if region_words is not None:
            slot['region_set'] = self.add_set(region_words)
        self.slot_recs.append(_SLOT_PACK(*_SLOT_FIELDS(slot)))
        self.slot_qbase.append(0)
        self.slot_cost.extend((slot['hours'], slot['node_mult'],
                               slot['time_value']))
        return len(self.slot_recs) - 1

    def add_task(self,
                 slot_begin: int,
                 slot_end: int,
                 parents: Sequence[int] = (),
                 edge_tariffs: Sequence[Sequence[float]] = (),
                 src_tariff: Optional[Sequence[float]] = None) -> int:
        n_clouds = len(self.store.clouds)
        n_parents = len(parents)
        parent_begin = len(self.parents)
        edge_begin = len(self.tariffs)
        src_begin = -1
        # (parents are ints and tariff rows lists of floats already: the
        # callers build them; no per-element conversion here)
        self.parents.extend(parents)
        assert len(edge_tariffs) == n_parents
        tariffs = self.tariffs
        for row in edge_tariffs:
            assert len(row) == n_clouds
            tariffs.extend(row)
        if src_tariff is not None:
            assert len(src_tariff) == n_clouds
            src_begin = len(tariffs)
            tariffs.extend(src_tariff)
        self.tasks.append({
            'slot_begin': slot_begin, 'slot_end': slot_end,
            'n_parents': n_parents, 'parent_begin': parent_begin,
            'edge_tariff_begin': edge_begin, 'src_tariff_begin': src_begin
        })
        self.task_recs.append(_TASK_PACK(slot_begin, slot_end, n_parents,
                                         parent_begin, edge_begin, src_begin))
        return len(self.tasks) - 1

    def set_task_field(self, i: int, name: str, value: int) -> None:
        self.tasks[i][name] = value
        self.task_recs[i] = _TASK_PACK(*_TASK_FIELDS(self.tasks[i]))

    def add_blocked(self, **fields) -> int:
        entry = {
            'cloud': -1, 'inst_id': -1, 'region_id': -1, 'zone_id': -1,
            'acc_key': -1, 'use_spot': -1
        }
        entry.update(fields)
        self.blocked.append(entry)
        return len(self.blocked) - 1

    def add_dag(self, task_begin: int, task_end: int, is_chain: bool,
                minimize_cost: bool, blocked_begin: int = 0,
                blocked_end: int = 0) -> int:
        self.dags.append({
            'task_begin': task_begin, 'task_end': task_end,
            'is_chain': int(is_chain), 'minimize_cost': int(minimize_cost),
            'blocked_begin': blocked_begin, 'blocked_end': blocked_end
        })
        return len(self.dags) - 1

    # -- packing ------------------------------------------------------------
    @staticmethod
    def _pack(rows: List[Dict[str, Any]], dtype: np.dtype) -> np.ndarray:
        arr = np.zeros(max(len(rows), 1), dtype=dtype)
        names = [n for n in dtype.names if n != 'pad_']
        for name in names:
            default = -1 if name in ('acc_set', 'fuzzy_set', 'region_id',
                                     'zone_id') else 0
            arr[name][:len(rows)] = [r.get(name, default) for r in rows]
        return arr

    def pack(self) -> 'PackedProblem':
        return PackedProblem(self)


def _apply_local_disk(spec: Dict[str, Any], local_disk: Optional[str]) -> None:
    """AWS local-disk filter (sky/catalog/common.py:481-506)."""
    if local_disk is None:
        return
    mode, size, at_least = resources_utils.parse_local_disk_str(
        local_disk.lower())
    if mode not in ('nvme', 'ssd'):
        raise ValueError('Local disk should be either nvme or ssd. '
                         f'Got {local_disk}.')
    spec['flags_require'] = spec.get('flags_require', 0) | _native.F_SSD
    if mode == 'nvme':
        spec['flags_require'] |= _native.F_NVME
    spec['disk_op'] = _native.DISK_GE if at_least else _native.DISK_NEAR
    spec['disk_size'] = float(size)


class PackedProblem:
    """numpy arrays + the ctypes view over them."""

    def __init__(self, b: ProblemBuilder):
        self.store = b.store
        self.n_queries = b.n_queries
        self.queries = (np.frombuffer(b''.join(b.query_recs),
                                      dtype=_native.QUERY_DTYPE)
                        if b.query_recs else np.zeros(
                            1, dtype=_native.QUERY_DTYPE))
        sets = set_table(b.store)
        self.n_sets = len(sets) // _native.ACC_SET_WORDS
        self.acc_sets = sets if len(sets) else np.zeros(
            _native.ACC_SET_WORDS, dtype=np.uint32)
        self.n_slots = b.n_slots
        if b.slot_recs:
            slots = np.frombuffer(b''.join(b.slot_recs),
                                  dtype=_native.SLOT_DTYPE).copy()
            qbase = np.asarray(b.slot_qbase, dtype=np.int32)
            for name in ('query', 'gate_query'):
                col = slots[name]
                col += qbase * (col >= 0)
            cost = np.asarray(b.slot_cost, dtype=np.float64).reshape(-1, 3)
            slots['hours'] = cost[:, 0]
            slots['node_mult'] = cost[:, 1]
            slots['time_value'] = cost[:, 2]
            self.slots = slots
        else:
            self.slots = np.zeros(1, dtype=_native.SLOT_DTYPE)
        self.tasks = (np.frombuffer(b''.join(b.task_recs),
                                    dtype=_native.TASK_DTYPE)
                      if b.task_recs else np.zeros(1, _native.TASK_DTYPE))
        self.n_tasks = len(b.tasks)
        self.parents = np.asarray(b.parents or [0], dtype=np.int32)
        self.n_parents = len(b.parents)
        self.tariffs = np.asarray(b.tariffs or [0.0], dtype=np.float64)
        self.n_tariffs = len(b.tariffs)
        self.blocked = ProblemBuilder._pack(b.blocked, _native.BLOCKED_DTYPE)
        self.n_blocked = len(b.blocked)
        self.dags = ProblemBuilder._pack(b.dags, _native.DAG_DTYPE)
        self.n_dags = len(b.dags)
        if b.reservations is not None and b.reservations[1] > 0:
            self.reservations, self.n_reservations = b.reservations
        else:
            self.reservations, self.n_reservations = None, 0

    def c_problem(self) -> _native.Problem:
        p = _native.Problem()
        p.queries = _addr(self.queries)
        p.n_queries = self.n_queries
        p.acc_sets = _addr(self.acc_sets)
        p.n_acc_sets = self.n_sets
        p.slots = _addr(self.slots)
        p.n_slots = self.n_slots
        p.tasks = _addr(self.tasks)
        p.n_tasks = self.n_tasks
        p.parents = _addr(self.parents)
        p.n_parents = self.n_parents
        p.tariffs = _addr(self.tariffs)
        p.n_tariffs = self.n_tariffs
        p.blocked = _addr(self.blocked)
        p.n_blocked = self.n_blocked
        p.dags = _addr(self.dags)
        p.n_dags = self.n_dags
        p.reservations = (None if self.reservations is None else
                          _addr(self.reservations))
        p.n_reservations = self.n_reservations
        return p

    def h2d_bytes(self) -> int:
        return int(self.queries.nbytes * (self.n_queries > 0) +
                   self.acc_sets.nbytes * (self.n_sets > 0) +
                   self.slots.nbytes + self.tasks.nbytes +
                   self.parents.nbytes + self.tariffs.nbytes +
                   self.blocked.nbytes * (self.n_blocked > 0) +
                   self.dags.nbytes +
                   16 * self.n_reservations)


class Solution:
    """Outputs of skyopt_optimize as numpy arrays."""

    def __init__(self, packed: PackedProblem, want_tables: bool,
                 table_cap: int = 0, want_scan: bool = False):
        self.packed = packed
        # per-query scan results cost an extra kernel; only on request
        self.scan = (np.zeros(max(packed.n_queries, 1),
                              dtype=_native.SCAN_RESULT_DTYPE)
                     if want_scan else None)
        self.slot_count = np.zeros(max(packed.n_slots, 1), dtype=np.int32)
        self.slot_inst = np.zeros(max(packed.n_slots, 1), dtype=np.int32)
        self.chosen = np.zeros(max(packed.n_tasks, 1),
                               dtype=_native.CANDIDATE_DTYPE)
        self.chosen_index = np.zeros(max(packed.n_tasks, 1), dtype=np.int32)
        self.task_n = np.zeros(max(packed.n_tasks, 1), dtype=np.int32)
        self.dag = np.zeros(max(packed.n_dags, 1),
                            dtype=_native.DAG_RESULT_DTYPE)
        self.tables: Optional[np.ndarray] = None
        self.table_offsets: Optional[np.ndarray] = None
        if want_tables:
            cap = table_cap or max(
                1, packed.n_slots * max(packed.store.max_group_rows, 1))
            self.tables = np.zeros(cap, dtype=_native.CANDIDATE_DTYPE)
            self.table_offsets = np.zeros(packed.n_tasks + 1, dtype=np.int64)
        self.stats = _native.Stats()

    def c_solution(self) -> _native.Solution:
        s = _native.Solution()
        s.scan = None if self.scan is None else _addr(self.scan)
        s.slot_count = _addr(self.slot_count)
        s.slot_inst = _addr(self.slot_inst)
        s.chosen = _addr(self.chosen)
        s.chosen_index = _addr(self.chosen_index)
        s.task_n_candidates = _addr(self.task_n)
        s.dag = _addr(self.dag)
        if self.tables is not None:
            s.candidates = _addr(self.tables)
            s.cand_cap = len(self.tables)
            s.task_cand_offset = _addr(self.table_offsets)
        else:
            s.candidates = None
            s.cand_cap = 0
            s.task_cand_offset = None
        return s

    def d2h_bytes(self) -> int:
        p = self.packed
        return int(p.n_queries * 20 + p.n_slots * 8 + p.n_tasks *
                   (_native.CANDIDATE_DTYPE.itemsize + 8) + p.n_dags * 16)

    def task_table(self, task: int) -> np.ndarray:
        assert self.tables is not None
        return self.tables[self.table_offsets[task]:self.table_offsets[task +
                                                                        1]]


def solve(builder: ProblemBuilder,
          device: int = 0,
          want_tables: bool = False) -> Solution:
    """One `skyopt_optimize` call for everything the builder holds."""
    packed = builder.pack()
    sol = Solution(packed, want_tables)
    lib = _native.load()
    handle = builder.store.handle(device)
    if packed.n_slots == 0:
        # Host rules (feature gates, unknown names) left nothing to ask the
        # device: every task is without candidates.
        sol.dag['status'][:] = 1
        for d in range(packed.n_dags):
            sol.dag['task_fail'][d] = 0
        sol.dag['objective'][:] = math.nan
        sol.chosen_index[:] = -1
        return sol
    prob = packed.c_problem()
    csol = sol.c_solution()
    _native.check(
        lib.skyopt_optimize(handle, ctypes.byref(prob), ctypes.byref(csol),
                            ctypes.byref(sol.stats)))
    global LAST_STATS  # pylint: disable=global-statement
    LAST_STATS = sol.stats
    timeline.device_event('skyopt_optimize', sol.stats)
    return sol


# SkyoptStats of the most recent solve() in this process (tests / tracing).
LAST_STATS = None


class Session:
    """`skyopt_session_*`: one full solve, then re-solves under a new blocked
    list with the candidate sets kept on the device (failover loop)."""

    def __init__(self, builder: ProblemBuilder, device: int = 0,
                 want_tables: bool = False):
        self.builder = builder
        self.want_tables = want_tables
        self._lib = _native.load()
        self._handle = ctypes.c_void_p()
        self.packed = builder.pack()
        if self.packed.n_slots == 0:
            raise ValueError('a session needs at least one slot')
        self.solution = Solution(self.packed, want_tables)
        prob = self.packed.c_problem()
        csol = self.solution.c_solution()
        _native.check(
            self._lib.skyopt_session_open(builder.store.handle(device),
                                          ctypes.byref(prob),
                                          ctypes.byref(csol),
                                          ctypes.byref(self.solution.stats),
                                          ctypes.byref(self._handle)))
        # the native session holds the catalog handle: the store closes its
        # open sessions before it destroys the handle (CatalogStore.close)
        self._store = builder.store
        builder.store.register_session(self)

    def resolve(self, blocked: List[Dict[str, int]]) -> Solution:
        """Re-masks and re-solves; `blocked` are `add_blocked`-style dicts."""
        if not self._handle:
            raise RuntimeError('session is closed')
        rows = ProblemBuilder._pack(blocked, _native.BLOCKED_DTYPE)  # pylint: disable=protected-access
        sol = Solution(self.packed, self.want_tables)
        csol = sol.c_solution()
        _native.check(
            self._lib.skyopt_session_resolve(
                self._handle, _addr(rows) if len(blocked) else None,
                len(blocked), ctypes.byref(csol), ctypes.byref(sol.stats)))
        self.solution = sol
        return sol

    def close(self) -> None:
        if self._handle:
            self._lib.skyopt_session_close(self._handle)
            self._handle = ctypes.c_void_p()
            self._store.unregister_session(self)

    def __del__(self):
        try:
            self.close()
        except Exception:  # pylint: disable=broad-except
            pass


def solve_timed(builder: ProblemBuilder, iters: int, flush_l2: bool = True,
                device: int = 0):
    """Device-resident timing loop (bench.py): per-iteration kernel times."""
    packed = builder.pack()
    sol = Solution(packed, False)
    lib = _native.load()
    handle = builder.store.handle(device)
    prob = packed.c_problem()
    csol = sol.c_solution()
    iter_ms = np.zeros(iters, dtype=np.float32)
    scan_ms = np.zeros(iters, dtype=np.float32)
    _native.check(
        lib.skyopt_optimize_timed(handle, ctypes.byref(prob),
                                  ctypes.byref(csol), iters, int(flush_l2),
                                  _addr(iter_ms), _addr(scan_ms),
                                  ctypes.byref(sol.stats)))
    return sol, iter_ms, scan_ms


class ScanOutput:

    def __init__(self, results, list_ids, list_prices, fuzzy_keys,
                 fuzzy_prices, stats):
        self.results = results
        self.list_ids = list_ids
        self.list_prices = list_prices
        self.fuzzy_keys = fuzzy_keys
        self.fuzzy_prices = fuzzy_prices
        self.stats = stats

    def instance_list(self, q: int) -> List[int]:
        n = int(self.results['n_list'][q])
        return [int(v) for v in self.list_ids[q, :n]]

    def fuzzy_list(self, q: int) -> List[int]:
        n = int(self.results['n_fuzzy'][q])
        return [int(v) for v in self.fuzzy_keys[q, :n]]


def scan(builder: ProblemBuilder,
         list_cap: int = 0,
         fuzzy_cap: int = 0,
         device: int = 0) -> ScanOutput:
    """`skyopt_scan`: filter + argmin (+ sorted tables) for the queries."""
    packed = builder.pack()
    n = packed.n_queries
    assert n > 0
    lib = _native.load()
    handle = builder.store.handle(device)
    results = np.zeros(n, dtype=_native.SCAN_RESULT_DTYPE)
    list_ids = list_prices = fuzzy_keys = fuzzy_prices = None
    if list_cap:
        list_ids = np.full((n, list_cap), -1, dtype=np.int32)
        list_prices = np.full((n, list_cap), math.nan, dtype=np.float64)
    if fuzzy_cap:
        fuzzy_keys = np.full((n, fuzzy_cap), -1, dtype=np.int32)
        fuzzy_prices = np.full((n, fuzzy_cap), math.nan, dtype=np.float64)
    stats = _native.Stats()
    _native.check(
        lib.skyopt_scan(handle, _addr(packed.queries), n,
                        _addr(packed.acc_sets), packed.n_sets,
                        _addr(results), _native.ptr(list_ids),
                        _native.ptr(list_prices), list_cap,
                        _native.ptr(fuzzy_keys), _native.ptr(fuzzy_prices),
                        fuzzy_cap, ctypes.byref(stats)))
    return ScanOutput(results, list_ids, list_prices, fuzzy_keys,
                      fuzzy_prices, stats)


def solve_tables(store: CatalogStore, values: Sequence[Sequence[float]],
                 clouds: Sequence[Sequence[int]],
                 parents: Sequence[Sequence[int]],
                 edge_tariffs: Sequence[Sequence[Sequence[float]]],
                 src_tariffs: Sequence[Optional[Sequence[float]]],
                 is_chain: bool, minimize_cost: bool,
                 device: int = 0) -> Tuple[List[int], float, int]:
    """`skyopt_solve_tables`: chain DP / exact DAG search on candidate tables
    the caller supplies (one DAG). Returns (chosen index per task, objective,
    status)."""
    n_tasks = len(values)
    n_clouds = len(store.clouds)
    offsets = np.zeros(n_tasks + 1, dtype=np.int64)
    for t, v in enumerate(values):
        offsets[t + 1] = offsets[t] + len(v)
    flat_v = np.ascontiguousarray(
        np.concatenate([np.asarray(v, dtype=np.float64) for v in values])
        if offsets[-1] else np.zeros(1))
    flat_c = np.ascontiguousarray(
        np.concatenate([np.asarray(c, dtype=np.int32) for c in clouds])
        if offsets[-1] else np.zeros(1, dtype=np.int32))
    tasks = np.zeros(n_tasks, dtype=_native.TASK_DTYPE)
    par: List[int] = []
    tar: List[float] = []
    for t in range(n_tasks):
        tasks['n_parents'][t] = len(parents[t])
        tasks['parent_begin'][t] = len(par)
        tasks['edge_tariff_begin'][t] = len(tar)
        tasks['src_tariff_begin'][t] = -1
        par.extend(int(p) for p in parents[t])
        for row in edge_tariffs[t]:
            assert len(row) == n_clouds
            tar.extend(float(x) for x in row)
        if src_tariffs[t] is not None:
            tasks['src_tariff_begin'][t] = len(tar)
            tar.extend(float(x) for x in src_tariffs[t])
    par_a = np.asarray(par or [0], dtype=np.int32)
    tar_a = np.asarray(tar or [0.0], dtype=np.float64)
    dags = np.zeros(1, dtype=_native.DAG_DTYPE)
    dags['task_end'] = n_tasks
    dags['is_chain'] = int(is_chain)
    dags['minimize_cost'] = int(minimize_cost)
    chosen = np.zeros(n_tasks, dtype=np.int32)
    results = np.zeros(1, dtype=_native.DAG_RESULT_DTYPE)
    lib = _native.load()
    _native.check(
        lib.skyopt_solve_tables(store.handle(device), _addr(flat_v),
                                _addr(flat_c), _addr(offsets),
                                _addr(tasks), n_tasks,
                                _addr(par_a), len(par),
                                _addr(tar_a), len(tar),
                                _addr(dags), 1, _addr(chosen),
                                _addr(results)))
    return ([int(i) for i in chosen], float(results['objective'][0]),
            int(results['status'][0]))
