"""Cloud base class: the feasibility API the optimizer drives.

Mirrors the placement-relevant surface of sky/clouds/cloud.py (Region / Zone
:77-92, CloudImplementationFeatures :33-62, get_feasible_launchable_resources
:459-501, check_features_are_supported :712-762, DummyCloud :1030-1033,
cloud_in_iterable :1037-1039). Provisioning, credentials, images, ... are out
of scope (SURVEY.md section 2b).

What is new: `plan_feasible()` states a request against this cloud as catalog
*queries* and an expansion *slot* for the GPU (engine.ProblemBuilder) instead
of running pandas filters. `get_feasible_launchable_resources()` and the fused
optimizer share that single description.
"""
import collections
import enum
from typing import Any, Callable, Dict, Iterable, List, Optional, Set, Tuple

from skypilot_b200 import _native
from skypilot_b200 import exceptions
from skypilot_b200.utils import resources_utils


_LATE: Dict[str, Any] = {}


def _late(name: str):
    """A sibling module that imports this one (resolved on first use; a
    function-level `from ... import` costs a microsecond per call and these
    sit in the per-request statement path)."""
    mod = _LATE.get(name)
    if mod is None:
        import importlib  # pylint: disable=import-outside-toplevel
        mod = importlib.import_module(f'skypilot_b200.{name}')
        _LATE[name] = mod
    return mod


class CloudImplementationFeatures(enum.Enum):
    STOP = 'stop'
    MULTI_NODE = 'multi-node'
    CLONE_DISK_FROM_CLUSTER = 'clone_disk_from_cluster'
    IMAGE_ID = 'image_id'
    DOCKER_IMAGE = 'docker_image'
    SPOT_INSTANCE = 'spot_instance'
    CUSTOM_DISK_TIER = 'custom_disk_tier'
    CUSTOM_NETWORK_TIER = 'custom_network_tier'
    OPEN_PORTS = 'open_ports'
    STORAGE_MOUNTING = 'storage_mounting'
    HOST_CONTROLLERS = 'host_controllers'
    HIGH_AVAILABILITY_CONTROLLERS = 'high_availability_controllers'
    AUTO_TERMINATE = 'auto_terminate'
    AUTOSTOP = 'autostop'
    AUTODOWN = 'autodown'
    CUSTOM_MULTI_NETWORK = 'custom_multi_network'
    LOCAL_DISK = 'local_disk'


class CloudCapability(str, enum.Enum):
    COMPUTE = 'compute'
    STORAGE = 'storage'


class Region(collections.namedtuple('Region', ['name'])):
    """A region with an optional ordered zone list."""
    name: str
    zones: Optional[List['Zone']] = None

    def set_zones(self, zones: List['Zone']):
        self.zones = zones
        for zone in self.zones:
            zone.region = self
        return self


class Zone(collections.namedtuple('Zone', ['name'])):
    name: str
    region: Region


class SlotPlan:
    """How one (request, cloud) pair is answered by the device."""

    def __init__(self):
        self.slot: Optional[int] = None      # builder slot, None = infeasible
        self.list_query: Optional[int] = None  # query naming instance types
        self.fuzzy_query: Optional[int] = None
        self.gate_query: Optional[int] = None
        self.hint: Optional[str] = None
        self.explicit_instance: Optional[str] = None
        self.no_fuzzy_when_matched = False
        # (instance type name, requested Resources) -> launchable Resources
        # (without region / zone); takes the request as an argument so that a
        # cached plan can serve any Resources object with the same fields
        self.make: Optional[Callable[[str, Any], Any]] = None


_INF = float('inf')


class _Recorded:
    """The records of one stated (request, cloud) pair: what plan_cached
    replays into a ProblemBuilder."""
    __slots__ = ('query_recs', 'slot_recs')

    def __init__(self):
        self.query_recs: List[bytes] = []
        self.slot_recs: List[bytes] = []

    @staticmethod
    def add_set(store, words) -> int:
        engine = _late('engine')
        by_obj = store.__dict__.setdefault('_set_id_by_obj', {})
        hit = by_obj.get(id(words))
        if hit is not None and hit[0] is words:
            return hit[1]
        return engine.ProblemBuilder(store).add_set(words)


class Cloud:
    """A cloud whose offerings live in the GPU-resident catalog."""

    _REPR = '<Cloud>'
    _CATALOG = ''  # key of the cloud in the catalog store
    _CLOUD_UNSUPPORTED_FEATURES: Dict[CloudImplementationFeatures, str] = {}
    # the name in the feature-gate message when it is not _REPR (the reference's
    # Shadeform prints the base class's '<Cloud>' there)
    _FEATURES_REPR: Optional[str] = None

    # ---- identity ---------------------------------------------------------
    def __repr__(self):
        return self._REPR

    def is_same_cloud(self, other: 'Cloud') -> bool:
        return isinstance(other, self.__class__)

    @classmethod
    def display_name(cls) -> str:
        return cls._REPR

    @classmethod
    def canonical_name(cls) -> str:
        return cls.__name__.lower()

    # ---- catalog plumbing ---------------------------------------------------
    @classmethod
    def _view(cls):
        return _late('catalog').view(cls._CATALOG)

    @classmethod
    def _rules(cls):
        return _late('catalog.rules').rules_for(cls._CATALOG)

    @classmethod
    def _catalog_module(cls):
        return _late('catalog').module_for(cls._CATALOG)

    # ---- regions / zones ----------------------------------------------------
    @classmethod
    def regions_with_offering(cls, instance_type: str,
                              accelerators: Optional[Dict[str, int]],
                              use_spot: bool, region: Optional[str],
                              zone: Optional[str],
                              resources: Optional[Any] = None) -> List[Region]:
        del accelerators, resources
        regions = cls._catalog_module().get_region_zones_for_instance_type(
            instance_type, use_spot)
        if region is not None:
            regions = [r for r in regions if r.name == region]
        if zone is not None:
            for r in regions:
                assert r.zones is not None, r
                r.set_zones([z for z in r.zones if z.name == zone])
            regions = [r for r in regions if r.zones]
        return regions

    @classmethod
    def optimize_by_zone(cls) -> bool:
        return False

    def validate_region_zone(
            self, region: Optional[str],
            zone: Optional[str]) -> Tuple[Optional[str], Optional[str]]:
        return self._catalog_module().validate_region_zone(region, zone)

    # ---- prices -------------------------------------------------------------
    def instance_type_to_hourly_cost(self, instance_type: str, use_spot: bool,
                                     region: Optional[str] = None,
                                     zone: Optional[str] = None) -> float:
        return self._catalog_module().get_hourly_cost(instance_type,
                                                      use_spot=use_spot,
                                                      region=region, zone=zone)

    def accelerators_to_hourly_cost(self, accelerators: Dict[str, int],
                                    use_spot: bool,
                                    region: Optional[str] = None,
                                    zone: Optional[str] = None) -> float:
        del accelerators, use_spot, region, zone
        return 0

    def get_egress_cost(self, num_gigabytes: float) -> float:
        del num_gigabytes
        return 0.0

    # ---- instance metadata --------------------------------------------------
    def instance_type_exists(self, instance_type: str) -> bool:
        return self._catalog_module().instance_type_exists(instance_type)

    @classmethod
    def get_vcpus_mem_from_instance_type(
            cls, instance_type: str) -> Tuple[Optional[float], Optional[float]]:
        return cls._catalog_module().get_vcpus_mem_from_instance_type(
            instance_type)

    @classmethod
    def get_accelerators_from_instance_type(
            cls, instance_type: str) -> Optional[Dict[str, Any]]:
        return cls._catalog_module().get_accelerators_from_instance_type(
            instance_type)

    @classmethod
    def get_default_instance_type(cls, cpus=None, memory=None, disk_tier=None,
                                  local_disk=None, region=None, zone=None,
                                  use_spot=False,
                                  max_hourly_cost=None) -> Optional[str]:
        return cls._catalog_module().get_default_instance_type(
            cpus=cpus, memory=memory, disk_tier=disk_tier,
            local_disk=local_disk, region=region, zone=zone,
            use_spot=use_spot, max_hourly_cost=max_hourly_cost)

    @classmethod
    def check_disk_tier(cls, instance_type: Optional[str],
                        disk_tier) -> Tuple[bool, str]:
        del instance_type, disk_tier
        return True, ''

    # ---- feature gate -------------------------------------------------------
    @classmethod
    def _unsupported_features_for_resources(
            cls, resources: Any,
            region: Optional[str] = None
    ) -> Dict[CloudImplementationFeatures, str]:
        del resources, region
        return dict(cls._CLOUD_UNSUPPORTED_FEATURES)

    @classmethod
    def check_features_are_supported(
            cls, resources: Any,
            requested_features: Set[CloudImplementationFeatures],
            region: Optional[str] = None) -> None:
        """Raises NotSupportedError naming the unsupported features
        (sky/clouds/cloud.py:712-762)."""
        unsupported = cls._unsupported_features_for_resources(
            resources, region)
        hit = requested_features.intersection(set(unsupported.keys()))
        if hit:
            rows = '\n\t'.join(f'{f.value} | {unsupported[f]}' for f in hit)
            raise exceptions.NotSupportedError(
                f'The following features are not supported by '
                f'{cls._FEATURES_REPR or cls._REPR}:'
                f'\n\tFeature | Reason\n\t{rows}')

    # ---- images --------------------------------------------------------------
    # Size of a cloud's stock images in GB: what the reference answers for a
    # `skypilot:` tag and when no credentials are present
    # (sky/clouds/aws.py:59, :547-569; sky/clouds/gcp.py:96, :405-422).
    _DEFAULT_IMAGE_GB = 0

    @classmethod
    def is_image_tag_valid(cls, image_tag: str, region: Optional[str]) -> bool:
        """sky/clouds/cloud.py is_image_tag_valid: <cloud>/images.csv."""
        return _late('catalog').is_image_tag_valid(image_tag, region,
                                                   clouds=cls._CATALOG)

    @classmethod
    def get_image_size(cls, image_id: str, region: Optional[str]) -> float:
        """GB of the image. The size of a custom image is a cloud API call in
        the reference; offline it answers the stock size, as the reference
        does without credentials."""
        del image_id, region
        return cls._DEFAULT_IMAGE_GB

    def _check_instance_type_accelerators_combination(self,
                                                      resources: Any) -> None:
        del resources

    def _feature_hint(self, resources: Any, num_nodes: int) -> Optional[str]:
        if resources.is_launchable():
            self._check_instance_type_accelerators_combination(resources)
        required = resources.get_required_cloud_features()
        if num_nodes > 1:
            required.add(CloudImplementationFeatures.MULTI_NODE)
        if not required:
            return None  # nothing asked for, nothing to refuse
        try:
            self.check_features_are_supported(resources, required)
        except exceptions.NotSupportedError as e:
            return str(e)
        return None

    # ---- feasibility ----------------------------------------------------------
    def get_feasible_launchable_resources(
            self, resources: Any,
            num_nodes: int = 1) -> resources_utils.FeasibleResources:
        """Offerings of this cloud that satisfy `resources`
        (sky/clouds/cloud.py:459-501): feature gate, then the catalog filter
        -- here one `skyopt_scan` call instead of pandas passes."""
        engine = _late('engine')
        hint = self._feature_hint(resources, num_nodes)
        if hint is not None:
            return resources_utils.FeasibleResources([], [], hint)
        view = self._view()
        b = engine.ProblemBuilder(view.store)
        plan = self.plan_feasible(b, resources, want_list=True)
        if plan.slot is None and plan.list_query is None and (
                plan.explicit_instance is None):
            fuzzy: List[str] = []
            if plan.fuzzy_query is not None:
                out = engine.scan(b, fuzzy_cap=self._fuzzy_cap(view),
                                  device=view.device)
                if not out.results['any_stage1'][plan.fuzzy_query]:
                    fuzzy = engine.format_fuzzy(
                        view.store, out.fuzzy_list(plan.fuzzy_query))
            return self._nothing_feasible(resources, fuzzy, plan.hint)
        if plan.explicit_instance is not None:
            if plan.slot is None:
                return self._nothing_feasible(resources, [], plan.hint)
            return resources_utils.FeasibleResources(
                [plan.make(plan.explicit_instance, resources)], [], None)
        n_inst = max(len(view.table.inst_names), 1)
        out = engine.scan(b, list_cap=min(n_inst, 2048),
                          fuzzy_cap=self._fuzzy_cap(view), device=view.device)
        return self._feasible_from_scan(view, plan, out, resources)

    def feasible_begin(self, b, resources: Any, num_nodes: int = 1):
        """get_feasible_launchable_resources in two halves, for many requests
        in ONE scan: states the request into the shared builder `b` (fuzzy
        candidates wanted, instance-type lists not) and returns a function of
        the scan output that gives the FeasibleResources -- cheapest instance
        type only. Used where only hints, fuzzy candidates and "anything at
        all?" matter: the error texts of a batch (Optimizer.optimize_batch)."""
        hint = self._feature_hint(resources, num_nodes)
        if hint is not None:
            gated = resources_utils.FeasibleResources([], [], hint)
            return lambda out: gated
        view = self._view()
        plan = self.plan_feasible(b, resources, want_list=False,
                                  want_fuzzy=True)
        engine = _late('engine')

        def end(out):
            if plan.slot is None and plan.list_query is None and (
                    plan.explicit_instance is None):
                fuzzy: List[str] = []
                if (plan.fuzzy_query is not None and
                        not out.results['any_stage1'][plan.fuzzy_query]):
                    fuzzy = engine.format_fuzzy(
                        view.store, out.fuzzy_list(plan.fuzzy_query))
                return self._nothing_feasible(resources, fuzzy, plan.hint)
            if plan.explicit_instance is not None:
                if plan.slot is None:
                    return self._nothing_feasible(resources, [], plan.hint)
                return resources_utils.FeasibleResources(
                    [plan.make(plan.explicit_instance, resources)], [], None)
            return self._feasible_from_scan(view, plan, out, resources)

        return end

    @staticmethod
    def _fuzzy_cap(view) -> int:
        return min(max(len(view.store.acc_keys), 1), 2048)

    def _feasible_from_scan(self, view, plan: SlotPlan, out,
                            resources) -> resources_utils.FeasibleResources:
        engine = _late('engine')
        fuzzy: List[str] = []
        gate = plan.gate_query if plan.gate_query is not None else (
            plan.fuzzy_query)
        if gate is not None and not out.results['any_stage1'][gate]:
            fuzzy = engine.format_fuzzy(view.store, out.fuzzy_list(gate))
            return self._nothing_feasible(resources, fuzzy, None)
        q = plan.list_query
        res = out.results[q]
        names: List[str] = []
        if res['best_inst'] >= 0:
            if out.results['n_list'][q] > 0:
                names = [
                    view.store.inst_names[i] for i in out.instance_list(q)
                ]
            else:
                names = [view.store.inst_names[int(res['best_inst'])]]
        made = [plan.make(n, resources) for n in names]
        made = [m for m in made if m is not None]
        if not made:
            return self._nothing_feasible(resources, fuzzy, None)
        return resources_utils.FeasibleResources(made, fuzzy, None)

    def _nothing_feasible(self, resources: Any, fuzzy: List[str],
                          hint: Optional[str]
                         ) -> resources_utils.FeasibleResources:
        """The answer when no offering satisfies `resources`; a few clouds
        word their own hint here (seeweb.py:337-345, shadeform.py:365-369)."""
        del resources
        return resources_utils.FeasibleResources([], fuzzy, hint)

    @staticmethod
    def _request_key(resources: Any) -> tuple:
        """Every field of a request that plan_feasible / _feature_hint read.
        Resources are immutable by convention (sky/resources.py:132-134), so
        two requests with the same key get the same constraint vectors."""
        r = resources
        accs = r._accelerators  # pylint: disable=protected-access
        args = r.accelerator_args
        return (r.instance_type, r._cpus, r._memory,  # pylint: disable=protected-access
                None if accs is None else tuple(accs.items()),
                None if args is None else args.get('tpu_vm', True),
                r.use_spot, r.region, r.zone, r.disk_tier, r.network_tier,
                r.local_disk, r.max_hourly_cost,
                None if r.image_id is None else tuple(sorted(
                    (str(k), v) for k, v in r.image_id.items())),
                None if r.ports is None else tuple(r.ports),
                _late('skypilot_config').generation())

    def plan_cached(self, builder, resources: Any, num_nodes: int = 1,
                    cost: Tuple[float, float, float] = (1.0, 1.0, 3600.0)
                   ) -> Tuple[SlotPlan, Optional[int]]:
        """`_feature_hint` + `plan_feasible`, memoised per (cloud, request
        fields) on the catalog store and replayed into `builder`: the fused
        optimizer states the same request shapes over and over (failover
        re-optimisation, batches of DAGs), and the Python rule code is the
        dominant host cost once the row work is on the GPU.

        Returns the (shared, read-only) plan template and the index of the
        slot it added to `builder` (None: nothing to ask the device)."""
        store = builder.store
        d = resources.__dict__
        # {request key: {(cloud class, multi-node): template}} on the store;
        # the inner dict is pinned on the Resources object, so that the long
        # request key is built and hashed once per object
        local = d.get('_plan_templates')
        generation = _late('skypilot_config')._generation  # pylint: disable=protected-access
        if (local is None or local[0] is not store or
                local[2] != generation):
            rkey = d.get('_request_key')
            if rkey is None or rkey[-1] != generation:
                rkey = self._request_key(resources)
                d['_request_key'] = rkey
            cache = store.__dict__.get('_plan_cache')
            if cache is None:
                cache = store.__dict__['_plan_cache'] = {}
            by_cloud = cache.get(rkey)
            if by_cloud is None:
                by_cloud = cache[rkey] = {}
            local = (store, by_cloud, generation)
            d['_plan_templates'] = local
        key = (self.__class__, num_nodes > 1)
        tmpl = local[1].get(key)
        if tmpl is None:
            tmpl = self.plan_fast(store, resources, num_nodes)
            if tmpl is None:
                plan = SlotPlan()
                recorder = _late('engine').ProblemBuilder(store)
                plan.hint = self._feature_hint(resources, num_nodes)
                if plan.hint is None:
                    plan = self.plan_feasible(recorder, resources)
                tmpl = (plan, recorder)
            local[1][key] = tmpl
        plan, recorder = tmpl
        if plan.slot is None:
            return plan, None
        # replay: the recorded bytes, the query base of this copy and the
        # slot's (hours, node_mult, time_value)
        builder.slot_qbase.append(len(builder.query_recs))
        builder.query_recs.extend(recorder.query_recs)
        slots = builder.slot_recs
        slots.append(recorder.slot_recs[plan.slot])
        builder.slot_cost.extend(cost)
        return plan, len(slots) - 1

    # ---- the common request shapes, stated without the generic machinery ----
    # `plan_fast` writes the same bytes as `_feature_hint` + `plan_feasible`
    # for a request that only names accelerators or vCPUs / memory (plus spot,
    # region, zone, price cap) -- the shape of nearly every task -- with
    # positional struct packs instead of per-field dicts. Anything else
    # (instance type, image, disks, ports, TPUs, a feature the cloud lacks, a
    # SkyPilot config) returns None and takes the generic path. Equality of
    # the two paths is a CPU test over every fixture scenario
    # (tests/test_host_statement.py::test_fast_statement_is_byte_identical).
    _FAST_PLAN = True

    def _fast_ctx(self, store):
        ctxs = store.__dict__.setdefault('_fast_ctx', {})
        ctx = ctxs.get(self.__class__)
        if ctx is None:
            engine = _late('engine')
            rules = self._rules()
            table = self._view().table
            cloud_obj = self.__class__()
            keeps_memory = rules.make_keeps_memory
            check = self.check_disk_tier

            def make(instance_type: str, res):
                ok, _ = check(instance_type, res.disk_tier)
                if not ok:
                    return None
                if keeps_memory:
                    return res.copy(cloud=cloud_obj,
                                    instance_type=instance_type,
                                    accelerators=None, cpus=None)
                return res.copy(cloud=cloud_obj, instance_type=instance_type,
                                accelerators=None, cpus=None, memory=None)

            default_cpus = None
            if rules.default_cpus is not None:
                default_cpus = (f'{rules.default_cpus}'
                                if rules.default_cpus_exact else
                                f'{rules.default_cpus}+')
            ctx = {
                'rules': rules, 'table': table, 'engine': engine,
                'index': table.index,
                'has_zone': bool(table.has_zone_column),
                'by_zone_always': bool(self.optimize_by_zone()),
                'us_first': int(rules.us_regions_first),
                'premium': bool(self._needs_premium_disk(None)),
                'make': make, 'default_cpus': default_cpus,
                'qpack': engine._QUERY_PACK, 'spack': engine._SLOT_PACK,  # pylint: disable=protected-access
                'generic': (self.__class__.plan_feasible is Cloud.plan_feasible
                            or getattr(self.__class__, '_FAST_TEMPLATE_OK',
                                       False)),
            }
            ctxs[self.__class__] = ctx
        return ctx

    def plan_fast(self, store, resources: Any, num_nodes: int):
        r = resources
        if (not self._FAST_PLAN or r._instance_type is not None or  # pylint: disable=protected-access
                r._image_id is not None or r._local_disk is not None or  # pylint: disable=protected-access
                r._disk_tier is not None or r._network_tier is not None or  # pylint: disable=protected-access
                r._ports is not None or r._accelerator_args is not None or  # pylint: disable=protected-access
                _late('skypilot_config').has_config()):
            return None
        ctx = self._fast_ctx(store)
        if not ctx['generic']:
            return None
        use_spot = bool(r._use_spot)  # pylint: disable=protected-access
        if use_spot or num_nodes > 1:
            # the feature gate (only these two can be asked for here)
            unsupported = self._unsupported_features_for_resources(r, None)
            if ((use_spot and
                 CloudImplementationFeatures.SPOT_INSTANCE in unsupported) or
                (num_nodes > 1 and
                 CloudImplementationFeatures.MULTI_NODE in unsupported)):
                return None
        rules, table, engine = ctx['rules'], ctx['table'], ctx['engine']
        plan = SlotPlan()
        rec = _Recorded()
        if use_spot and not rules.supports_spot:
            return plan, rec
        no_slot = use_spot and rules.spot_without_regions
        plan.make = ctx['make']
        accelerators = r._accelerators  # pylint: disable=protected-access
        max_cost = r._max_hourly_cost  # pylint: disable=protected-access
        max_price = _INF if max_cost is None else float(max_cost)
        region, zone = r._region, r._zone  # pylint: disable=protected-access
        premium = ctx['premium']
        index = ctx['index']
        if accelerators is None:
            cpus, memory = r._cpus, r._memory  # pylint: disable=protected-access
            if (cpus is None and
                    (memory is None or rules.default_cpus_always) and
                    ctx['default_cpus'] is not None):
                cpus = ctx['default_cpus']
            if memory is None and rules.default_memory is not None:
                memory = rules.default_memory
            elif memory is None and rules.default_mem_ratio is not None:
                memory = f'{rules.default_mem_ratio}x'
            flags = (_native.F_DEFAULT_FAMILY | _native.F_HAS_INSTANCE |
                     (_native.F_PREMIUM_DISK if premium else 0))
            in_region = rules.default_query_region
            cop, cval = engine.parse_cpus(cpus)
            mop, mval = engine.parse_memory(memory)
            rec.query_recs.append(ctx['qpack'](
                index, 0, flags, 0, -1, -1,
                1 if (use_spot and max_cost is not None) else 0, cop, mop, 0,
                engine.region_filter_id(table, region if in_region else None),
                engine.zone_filter_id(table, zone if in_region else None),
                0, cval, mval, 0, max_price))
            plan.list_query = 0
        else:
            assert len(accelerators) == 1, resources
            acc, acc_count = next(iter(accelerators.items()))
            exact, _, _ = engine.accelerator_sets(store, acc, acc_count)
            in_region = rules.acc_query_region
            cop, cval = engine.parse_cpus(
                r._cpus if rules.acc_query_cpus else None)  # pylint: disable=protected-access
            mop, mval = engine.parse_memory(
                r._memory if rules.acc_query_memory else None)  # pylint: disable=protected-access
            rec.query_recs.append(ctx['qpack'](
                index, _native.Q_ACC, 0, 0, rec.add_set(store, exact), -1,
                1 if (use_spot and not rules.spot_without_regions) else 0,
                cop, mop, 0,
                engine.region_filter_id(table, region if in_region else None),
                engine.zone_filter_id(table, zone if in_region else None),
                _native.F_PREMIUM_DISK if premium else 0, cval, mval, 0,
                max_price))
            plan.list_query = 0
            plan.fuzzy_query = 0
        if not no_slot:
            by_zone = ctx['has_zone'] and (use_spot or ctx['by_zone_always'])
            rec.slot_recs.append(ctx['spack'](
                index, 0, -1, -1, -1, 1 if use_spot else 0,
                engine.region_exact_id(table, region),
                engine.zone_exact_id(table, zone), int(by_zone),
                ctx['us_first'], -1, int(use_spot), -1, 1.0, 1.0, 3600.0))
            plan.slot = 0
        return plan, rec

    def plan_feasible(self, builder, resources: Any,
                      want_list: bool = False,
                      want_fuzzy: Optional[bool] = None) -> SlotPlan:
        """States `resources` against this cloud for the device: the template
        shared by AWS, Azure, Lambda and the other single-table clouds
        (aws.py:881-953, azure.py:485-557, lambda_cloud.py:217-280)."""
        store = builder.store
        ctxs = store.__dict__.setdefault('_plan_ctx', {})
        ctx = ctxs.get(self.__class__)
        if ctx is None:
            # what the statement needs of this cloud's table and rules: a
            # property of (catalog, cloud), looked up once
            rules = self._rules()
            table = self._view().table
            ctx = (rules, table, bool(table.has_zone_column), _late('engine'))
            ctxs[self.__class__] = ctx
        rules, table, has_zone_column, engine = ctx
        # read per call: AWS splits by zone while the config enables
        # reservations (the plan templates are keyed on the config generation)
        by_zone_always = bool(self.optimize_by_zone())
        plan = SlotPlan()
        use_spot = bool(resources.use_spot)
        if use_spot and not rules.supports_spot:
            return plan
        # IBM: the queries are stated, but a spot request gets no slot
        no_slot = use_spot and rules.spot_without_regions
        by_zone = has_zone_column and (use_spot or by_zone_always)
        slot_common = dict(
            cloud=table.index, price_col=1 if use_spot else 0,
            region_id=engine.region_exact_id(table, resources.region),
            zone_id=engine.zone_exact_id(table, resources.zone),
            split_by_zone=int(by_zone), us_first=int(rules.us_regions_first),
            use_spot=int(use_spot),
            region_words=region_allow_words(table, resources, self))

        if resources.instance_type is not None:
            ok, _ = self.check_disk_tier(resources.instance_type,
                                         resources.disk_tier)
            inst = table.inst_index.get(resources.instance_type, -1)
            plan.explicit_instance = resources.instance_type
            plan.make = lambda name, res: res.copy(accelerators=None)
            if ok and inst >= 0 and not no_slot:
                plan.slot = builder.add_slot(inst_id=inst, **slot_common)
            return plan

        cloud_obj = self.__class__()
        keeps_memory = rules.make_keeps_memory

        def make(instance_type: str, res):
            ok, _ = self.check_disk_tier(instance_type, res.disk_tier)
            if not ok:
                return None
            if keeps_memory:
                return res.copy(cloud=cloud_obj, instance_type=instance_type,
                                accelerators=None, cpus=None)
            return res.copy(cloud=cloud_obj, instance_type=instance_type,
                            accelerators=None, cpus=None, memory=None)

        plan.make = make
        premium = self._needs_premium_disk(resources.disk_tier)
        local_disk = (resources.local_disk
                      if rules.supports_local_disk else None)
        accelerators = resources.accelerators
        if accelerators is None:
            cpus, memory = resources.cpus, resources.memory
            if (cpus is None and
                    (memory is None or rules.default_cpus_always) and
                    rules.default_cpus is not None):
                cpus = (f'{rules.default_cpus}' if rules.default_cpus_exact
                    else f'{rules.default_cpus}+')
            if memory is None and rules.default_memory is not None:
                memory = rules.default_memory
            elif memory is None and rules.default_mem_ratio is not None:
                memory = f'{rules.default_mem_ratio}x'
            flags = _native.F_DEFAULT_FAMILY
            if premium:
                flags |= _native.F_PREMIUM_DISK
            q_region = resources.region if rules.default_query_region else None
            q_zone = resources.zone if rules.default_query_region else None
            spec = builder.cpus_mem_query(
                table, cpus, memory, q_region, q_zone,
                use_spot, resources.max_hourly_cost, flags_require=flags,
                local_disk=local_disk)
            q = builder.add_query(spec)
            plan.list_query = q
            if not no_slot:
                plan.slot = builder.add_slot(query=q, **slot_common)
            return plan

        assert len(accelerators) == 1, resources
        acc, acc_count = list(accelerators.items())[0]
        spec = builder.accelerator_query(
            table, acc, acc_count,
            resources.cpus if rules.acc_query_cpus else None,
            resources.memory if rules.acc_query_memory else None,
            use_spot and not rules.spot_without_regions,
            resources.region if rules.acc_query_region else None,
            resources.zone if rules.acc_query_region else None,
            resources.max_hourly_cost, local_disk=local_disk,
            flags_require2=_native.F_PREMIUM_DISK if premium else 0,
            want_list=want_list,
            want_fuzzy=want_list if want_fuzzy is None else want_fuzzy)
        q = builder.add_query(spec)
        plan.list_query = q
        plan.fuzzy_query = q
        if not no_slot:
            plan.slot = builder.add_slot(query=q, **slot_common)
        return plan

    @classmethod
    def _needs_premium_disk(cls, disk_tier) -> bool:
        del disk_tier
        return False

    # Object-path variant kept for API parity; the fused optimizer never
    # calls it.
    def _get_feasible_launchable_resources(
            self, resources: Any) -> resources_utils.FeasibleResources:
        return self.get_feasible_launchable_resources(resources)


def _exact_region(table, region: Optional[str]) -> int:
    engine = _late('engine')
    return engine.region_exact_id(table, region)


def _exact_zone(table, zone: Optional[str]) -> int:
    engine = _late('engine')
    return engine.zone_exact_id(table, zone)


class DummyCloud(Cloud):
    """Zero egress cost from / to; used for the optimizer's source / sink."""
    _REPR = 'DummyCloud'


def cloud_in_iterable(cloud: Cloud, cloud_list: Iterable[Cloud]) -> bool:
    cls = cloud.__class__
    for c in cloud_list:
        if c.__class__ is cls or cloud.is_same_cloud(c):
            return True
    return False


def region_allow_words(table, resources: Any, cloud_obj: Any):
    """Bitmask over the cloud's region ids of the regions a launchable of
    `resources` on this cloud may use, or None (every region): the per-region
    `image_id` dict and the per-region `ssh_proxy_command` of the SkyPilot
    config (Resources.get_valid_regions_for_launchable,
    sky/resources.py:1210-1246)."""
    image_id = resources.image_id
    config = _late('skypilot_config')
    if image_id is None and not config.has_config():
        return None
    import numpy as np  # pylint: disable=import-outside-toplevel
    names = None
    if image_id is not None and None not in image_id:
        names = set(image_id.keys())
    by_proxy = config.allowed_regions_by_ssh_proxy(str(cloud_obj).lower())
    if by_proxy is not None:
        names = by_proxy if names is None else names & by_proxy
    if names is None:
        return None
    words = np.zeros(_native.ACC_SET_WORDS, dtype=np.uint32)
    for name in names:
        rid = table.region_exact.get(name)
        if rid is not None and rid < 32 * _native.ACC_SET_WORDS:
            words[rid >> 5] |= np.uint32(1 << (rid & 31))
    return words
