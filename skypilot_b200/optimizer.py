"""The placement optimizer behind `Optimizer.optimize(dag)`.

Public surface and semantics follow sky/optimizer.py (Optimizer.optimize
:106-142, _optimize_dag :1381-1512, _estimate_nodes_cost_or_time :239-426,
_fill_in_launchable_resources :1664-1785, chain DP :429-487, general DAGs
:490-637, totals :640-698, egress :75-104 / :196-236). The inner loops do not
run here: `_solve()` states the whole DAG -- every (task, requested
Resources, cloud) feasibility filter, the region/zone expansion, per-candidate
cost, the blocked filter and the DP / exact search -- as ONE device problem
(engine.ProblemBuilder -> skyopt_optimize) and reads back the plan. Host code
keeps what is Python by nature: per-cloud rules, time-estimator callbacks,
egress tariffs (a few scalars per edge) and building the `Resources` objects
of the answer.
"""
import collections
import enum
import logging
import math
from typing import Any, Dict, Iterable, List, Optional, Tuple

import networkx as nx

from skypilot_b200 import catalog
from skypilot_b200 import check as sky_check
from skypilot_b200 import clouds
from skypilot_b200 import dag as dag_lib
from skypilot_b200 import engine
from skypilot_b200 import exceptions
from skypilot_b200 import reservations
from skypilot_b200 import resources as resources_lib
from skypilot_b200 import skypilot_config
from skypilot_b200 import task as task_lib
from skypilot_b200.utils import resources_utils
from skypilot_b200.utils import timeline

logger = logging.getLogger(__name__)

_DUMMY_SOURCE_NAME = 'skypilot-dummy-source'
_DUMMY_SINK_NAME = 'skypilot-dummy-sink'

_TaskToCostMap = Dict[task_lib.Task, Dict[resources_lib.Resources, float]]
_PerCloudCandidates = Dict[clouds.Cloud, List[resources_lib.Resources]]
_TaskToPerCloudCandidates = Dict[task_lib.Task, _PerCloudCandidates]


class OptimizeTarget(enum.Enum):
    COST = 0
    TIME = 1


class DummyResources(resources_lib.Resources):
    """Resources of the dummy source / sink: zero cost, zero egress."""
    _REPR = 'DummyResources'

    def __repr__(self) -> str:
        return DummyResources._REPR

    def get_cost(self, seconds):
        return 0


def _is_dummy(task: task_lib.Task) -> bool:
    return task.name in (_DUMMY_SOURCE_NAME, _DUMMY_SINK_NAME)


class _SlotInfo:
    """Host memo of one device slot: who asked, on which cloud, and how to
    turn the answer back into a Resources."""
    __slots__ = ('task', 'resources', 'cloud', 'plan', 'table')

    def __init__(self, task, resources, cloud, plan, table):
        self.task = task
        self.resources = resources
        self.cloud = cloud
        self.plan = plan
        self.table = table


class _Problem:
    """A DAG stated for the device plus what is needed to read the answer."""

    def __init__(self, builder, tasks, slot_info, hints, minimize_cost,
                 is_chain):
        self.builder = builder
        self.tasks: List[task_lib.Task] = tasks
        self.slot_info: List[_SlotInfo] = slot_info
        self.hints = hints
        self.minimize_cost = minimize_cost
        self.is_chain = is_chain
        self.solution: Optional[engine.Solution] = None

    def launchable(self, cand) -> resources_lib.Resources:
        """The launchable Resources of one device candidate record."""
        info = self.slot_info[int(cand['slot'])]
        inst = int(cand['inst_id'])
        name = 'TPU-VM' if inst == -2 else (
            self.builder.store.inst_names[inst])
        base = info.plan.make(name, info.resources)
        region = info.table.region_names[int(cand['region_id'])]
        zid = int(cand['zone_id'])
        zone = info.table.zone_names[zid] if zid >= 0 else None
        if base is info.resources:
            # the request itself (explicit instance type): never mutated
            if zone is not None:
                return base.copy(region=region, zone=zone)
            return base.copy(region=region)
        # `make` returned a fresh copy: place it without a second clone
        base._region = region  # pylint: disable=protected-access
        if zone is not None:
            base._zone = zone  # pylint: disable=protected-access
        return base


class Optimizer:
    """Assigns the best launchable Resources to every task of a DAG."""

    # ------------------------------------------------------------------ egress
    @staticmethod
    def _egress_cost(src_cloud: clouds.Cloud, dst_cloud: clouds.Cloud,
                     gigabytes: float) -> float:
        if isinstance(src_cloud, clouds.DummyCloud) or isinstance(
                dst_cloud, clouds.DummyCloud):
            return 0.0
        if not src_cloud.is_same_cloud(dst_cloud):
            return src_cloud.get_egress_cost(num_gigabytes=gigabytes)
        return 0.0

    @staticmethod
    def _egress_time(src_cloud: clouds.Cloud, dst_cloud: clouds.Cloud,
                     gigabytes: float) -> float:
        if isinstance(src_cloud, clouds.DummyCloud) or isinstance(
                dst_cloud, clouds.DummyCloud):
            return 0.0
        if not src_cloud.is_same_cloud(dst_cloud):
            bandwidth_gbps = 10  # sky/optimizer.py:97-101
            return gigabytes * 8 / bandwidth_gbps
        return 0.0

    @staticmethod
    def _get_egress_info(parent, parent_resources, node, resources):
        if isinstance(parent_resources.cloud, clouds.DummyCloud):
            if node.get_inputs() is None:
                return None, None, 0
            src_cloud = node.get_inputs_cloud()
            nbytes = node.get_estimated_inputs_size_gigabytes()
        else:
            src_cloud = parent_resources.cloud
            nbytes = parent.get_estimated_outputs_size_gigabytes()
        return src_cloud, resources.cloud, nbytes

    @staticmethod
    def _egress_cost_or_time(minimize_cost: bool, parent, parent_resources,
                             node, resources):
        src_cloud, dst_cloud, nbytes = Optimizer._get_egress_info(
            parent, parent_resources, node, resources)
        if not nbytes:
            return 0
        assert src_cloud is not None and dst_cloud is not None
        fn = Optimizer._egress_cost if minimize_cost else (
            Optimizer._egress_time)
        return fn(src_cloud, dst_cloud, nbytes)

    # -------------------------------------------------------------- public API
    @staticmethod
    @timeline.event
    def optimize(dag: 'dag_lib.Dag',
                 minimize: OptimizeTarget = OptimizeTarget.COST,
                 blocked_resources: Optional[Iterable[
                     resources_lib.Resources]] = None,
                 quiet: bool = False) -> 'dag_lib.Dag':
        """Finds the best execution plan and stores it in
        `task.best_resources` of every task (sky/optimizer.py:106-142).

        Raises:
            exceptions.ResourcesUnavailableError: a task has no candidate.
            exceptions.NoCloudAccessError: no cloud is enabled.
        """
        _check_specified_clouds(dag)
        if quiet:
            # The dummy source / sink only matter to the reference's Python DP
            # and to the totals of the printed plan: the device problem is
            # stated on the real tasks (a DAG is a chain with or without them,
            # Dag.is_chain), so a quiet call leaves the graph alone.
            Optimizer._optimize_dag(
                dag=dag,
                minimize_cost=minimize == OptimizeTarget.COST,
                blocked_resources=blocked_resources,
                quiet=True)
            return dag
        Optimizer._add_dummy_source_sink_nodes(dag)
        try:
            Optimizer._optimize_dag(
                dag=dag,
                minimize_cost=minimize == OptimizeTarget.COST,
                blocked_resources=blocked_resources,
                quiet=quiet)
        finally:
            Optimizer._remove_dummy_source_sink_nodes(dag)
        return dag

    @staticmethod
    def _add_dummy_source_sink_nodes(dag: 'dag_lib.Dag') -> None:
        """Source -> every root, every leaf -> Sink (sky/optimizer.py:145)."""
        graph = dag.get_graph()
        roots = [n for n, d in graph.in_degree() if d == 0]
        leaves = [n for n, d in graph.out_degree() if d == 0]

        def make_dummy(name):
            dummy = task_lib.Task(name)
            dummy.set_resources({DummyResources(cloud=clouds.DummyCloud())})
            dummy.set_time_estimator(lambda _: 0)
            return dummy

        with dag:
            source = make_dummy(_DUMMY_SOURCE_NAME)
            for node in roots:
                source >> node  # pylint: disable=pointless-statement
            sink = make_dummy(_DUMMY_SINK_NAME)
            for node in leaves:
                node >> sink  # pylint: disable=pointless-statement

    @staticmethod
    def _remove_dummy_source_sink_nodes(dag: 'dag_lib.Dag') -> None:
        source = [t for t in dag.tasks if t.name == _DUMMY_SOURCE_NAME]
        sink = [t for t in dag.tasks if t.name == _DUMMY_SINK_NAME]
        if not source and not sink:
            return
        assert len(source) == len(sink) == 1, dag.tasks
        dag.remove(source[0])
        dag.remove(sink[0])

    @staticmethod
    def optimize_batch(dags: List['dag_lib.Dag'],
                       minimize: OptimizeTarget = OptimizeTarget.COST,
                       blocked_resources: Optional[Iterable[
                           resources_lib.Resources]] = None,
                       devices: Optional[List[int]] = None,
                       return_exceptions: bool = False) -> List[Any]:
        """Optimizes independent DAGs together (BASELINE.json config 5).

        DAG *i* goes to GPU `devices[i % len(devices)]`; every GPU holds a
        replica of the catalog and solves its shard as ONE device problem
        (one H2D; four launches: expand, scan, gather, solve; one D2H), the
        shards run concurrently from one host thread per GPU. No collective is involved: the DAGs are
        independent (north_star: "no NCCL needed").

        Returns the DAGs (each task's `best_resources` set). A DAG without a
        feasible plan raises ResourcesUnavailableError, or -- with
        `return_exceptions` -- yields the exception object in its slot.
        """
        import threading  # pylint: disable=import-outside-toplevel
        minimize_cost = minimize == OptimizeTarget.COST
        blocked = list(blocked_resources or [])
        store = catalog.get_store()
        devices = list(devices) if devices else [catalog.get_device()]
        shards: List[List[int]] = [[] for _ in devices]
        for i in range(len(dags)):
            shards[i % len(devices)].append(i)
        problems: Dict[int, _Problem] = {}
        builders = [engine.ProblemBuilder(store) for _ in devices]
        first_task: Dict[int, int] = {}
        enabled = sky_check.get_cached_enabled_clouds_or_refresh(
            raise_if_no_cloud_access=True)
        for shard, b in zip(shards, builders):
            for i in shard:
                dag = dags[i]
                _check_specified_clouds(dag, enabled)
                choice = Optimizer._resolve_ordered_resources(dag, blocked)
                saved = {t: t.resources for t in choice}
                for t, c in choice.items():
                    t.resources = {c}
                try:
                    # The dummy source / sink of the single-DAG path only
                    # matter to the reference's Python DP; the device problem
                    # is stated on the real tasks (a DAG is a chain with the
                    # dummies attached iff it is one without them).
                    graph = dag.get_graph()
                    topo = (list(dag.tasks) if len(dag.tasks) == 1 else list(
                        nx.topological_sort(graph)))
                    first_task[i] = len(b.tasks)
                    problems[i] = Optimizer._state_problem(
                        graph, topo, minimize_cost, blocked, dag.is_chain(),
                        builder=b, enabled=enabled)
                finally:
                    for t, original in saved.items():
                        t.resources = original
        solutions: List[Optional[engine.Solution]] = [None] * len(devices)
        errors: List[Optional[BaseException]] = [None] * len(devices)

        def run(k: int) -> None:
            try:
                if builders[k].dags:
                    solutions[k] = engine.solve(builders[k], device=devices[k])
            except BaseException as e:  # pylint: disable=broad-except
                errors[k] = e

        threads = [threading.Thread(target=run, args=(k,))
                   for k in range(len(devices))]
        for th in threads:
            th.start()
        for th in threads:
            th.join()
        for e in errors:
            if e is not None:
                raise e
        out: List[Any] = [None] * len(dags)
        failed: List[Tuple[int, task_lib.Task]] = []
        for k, shard in enumerate(shards):
            sol = solutions[k]
            for d, i in enumerate(shard):
                problem = problems[i]
                res = sol.dag[d]
                try:
                    if res['status'] == 1:
                        task = problem.tasks[int(res['task_fail'])]
                        if return_exceptions:
                            failed.append((i, task))  # worded below, together
                            continue
                        Optimizer._raise_unavailable(task, blocked)
                    if res['status'] != 0:
                        # beyond the device enumeration: the single-DAG path
                        # solves it by elimination on the host
                        Optimizer.optimize(dags[i], minimize, blocked,
                                           quiet=True)
                        out[i] = dags[i]
                        continue
                    for j, task in enumerate(problem.tasks):
                        task.best_resources = problem.launchable(
                            sol.chosen[first_task[i] + j])
                    out[i] = dags[i]
                except exceptions.ResourcesUnavailableError as e:
                    if not return_exceptions:
                        raise
                    out[i] = e
        if failed:
            errors = Optimizer._unavailable_errors([t for _, t in failed])
            for (i, _), e in zip(failed, errors):
                out[i] = e
        return out

    # -------------------------------------------------------------- job groups
    @staticmethod
    @timeline.event
    def optimize_job_group(dag: 'dag_lib.Dag',
                           minimize: OptimizeTarget = OptimizeTarget.COST,
                           blocked_resources: Optional[Iterable[
                               resources_lib.Resources]] = None,
                           quiet: bool = False) -> 'dag_lib.Dag':
        """Places all jobs of a JobGroup on one (cloud, region)
        (sky/optimizer.py:1039-1200, :1265-1378).

        The candidate tables of every job come from ONE device call (the jobs
        are stated as independent single-task DAGs); the intersection of
        their (cloud, region) sets and the per-infra sums run on those tables.
        Without a common infra each job keeps its own optimum, like
        `_optimize_independent`.

        Where the reference is not deterministic this implementation is: its
        `_select_best_infra` looks the infra's Cloud *object* up in the other
        jobs' candidate dicts, and since every launchable carries a fresh
        `AWS()` / `GCP()` instance (aws.py:905) the look-up fails for all jobs
        but the first, every infra is discarded and `common_infras[0]` -- the
        first element of a Python set of strings -- is returned. Here the
        infra with the lowest total cost (or time) wins, ties by (cloud,
        region) order. With exactly one common infra, with one job, and
        without a common infra both agree.
        """
        if not dag.is_job_group():
            return Optimizer.optimize(dag, minimize, blocked_resources, quiet)
        minimize_cost = minimize == OptimizeTarget.COST
        blocked = list(blocked_resources or [])
        tasks = list(dag.tasks)
        _check_specified_clouds(dag)
        enabled = sky_check.get_cached_enabled_clouds_or_refresh(
            raise_if_no_cloud_access=True)
        store = catalog.get_store()
        b = engine.ProblemBuilder(store)
        problems = []
        ordered = Optimizer._resolve_ordered_resources(dag, blocked)
        saved = {t: t.resources for t in ordered}
        for t, c in ordered.items():
            t.resources = {c}
        try:
            for task in tasks:
                graph = nx.DiGraph()
                graph.add_node(task)
                problems.append(
                    Optimizer._state_problem(graph, [task], minimize_cost,
                                             blocked, True, builder=b,
                                             enabled=enabled))
        finally:
            for t, original in saved.items():
                t.resources = original
        sol = engine.solve(b, device=catalog.get_device(), want_tables=True)
        # per job: ordered candidates as (cloud index, region id, value, record)
        tables = []
        for i, task in enumerate(tasks):
            rows = sol.task_table(i) if sol.tables is not None else []
            if len(rows) == 0:
                raise exceptions.ResourcesUnavailableError(
                    f'No resources available for job "{task.name}" '
                    f'in JobGroup "{dag.name}"')
            cands = []
            for cand in rows:
                info = problems[i].slot_info[int(cand['slot'])]
                score = float(cand['value'])
                if task.time_estimator_func is not None:
                    # unlike the DAG path, the job-group score estimates the
                    # runtime on the launchable (sky/optimizer.py:1348-1361)
                    runtime = task.estimate_runtime(
                        problems[i].launchable(cand))
                    if runtime is None:
                        runtime = 3600
                    score = (float(float(cand['hourly']) * (runtime / 3600)) *
                             task.num_nodes if minimize_cost else runtime)
                cands.append((info.table.index, int(cand['region_id']), score,
                              cand))
            tables.append(cands)
        common = Optimizer._find_common_infras(tables)
        if not common:
            if not quiet:
                logger.warning('No common infrastructure found for all jobs. '
                               'Falling back to independent optimization.')
            for i, task in enumerate(tasks):
                task.best_resources = problems[i].launchable(sol.chosen[i])
            return dag
        best = Optimizer._select_best_infra(common, tables, store)
        cloud_idx, region_id = best
        for i, task in enumerate(tasks):
            for c, r, _, cand in tables[i]:
                if c == cloud_idx and r == region_id:
                    resources = problems[i].launchable(cand)
                    task.best_resources = resources
                    # keeps the constraint through re-serialisation
                    # (sky/optimizer.py:1182-1193)
                    task.set_resources_override({
                        'cloud': resources.cloud, 'region': resources.region
                    })
                    break
        if not quiet:
            table = store.clouds[cloud_idx]
            logger.info('Selected infrastructure: %s/%s', table.name,
                        table.region_names[region_id])
        return dag

    @staticmethod
    def _find_common_infras(tables) -> List[Tuple[int, int]]:
        """(cloud, region) pairs every job has a candidate in
        (sky/optimizer.py:1265-1313), in (cloud, region) order."""
        common = None
        for cands in tables:
            infras = {(c, r) for c, r, _, _ in cands}
            common = infras if common is None else common & infras
        return sorted(common or [])

    @staticmethod
    def _select_best_infra(common, tables, store) -> Tuple[int, int]:
        """Lowest sum over the jobs of their cheapest (or fastest) candidate
        on the infra (sky/optimizer.py:1315-1378)."""
        best, best_score = None, math.inf
        for infra in common:
            total = 0.0
            for cands in tables:
                total += min(v for c, r, v, _ in cands if (c, r) == infra)
            if total < best_score:
                best, best_score = infra, total
        del store
        return best if best is not None else common[0]

    # ---------------------------------------------------- problem construction
    @staticmethod
    def _runtime(task, n_resources: int, orig_resources) -> float:
        """Estimated runtime in seconds (sky/optimizer.py:320-339)."""
        if task.time_estimator_func is None:
            return 1 * 3600
        if n_resources == 1 and task.time_estimator_func is None:
            return 1 * 3600
        return task.estimate_runtime(orig_resources)

    @staticmethod
    def _state_problem(dag_graph,
                       topo_real: List[task_lib.Task],
                       minimize_cost: bool,
                       blocked_resources,
                       is_chain: bool,
                       builder: Optional[engine.ProblemBuilder] = None,
                       enabled: Optional[List[clouds.Cloud]] = None
                      ) -> _Problem:
        """States all real tasks of one DAG for the device."""
        if enabled is None:
            enabled = sky_check.get_cached_enabled_clouds_or_refresh(
                raise_if_no_cloud_access=True)
        store = catalog.get_store()
        b = builder if builder is not None else engine.ProblemBuilder(store)
        if b.reservations is None:
            # reserved capacity per (cloud, instance type, zone): one table
            # for every DAG stated into this builder
            b.reservations = reservations.device_table(store)
        n_clouds = len(store.clouds)
        cloud_objs = store.__dict__.get('_cloud_objs')
        if cloud_objs is None:
            cloud_objs = [_cloud_object(t.name) for t in store.clouds]
            store.__dict__['_cloud_objs'] = cloud_objs
        # enabled clouds that the catalog holds, with their tables
        tables = store.__dict__.setdefault('_tables_by_class', {})
        slot_info: List[_SlotInfo] = [None] * b.n_slots  # type: ignore
        hints: Dict[Any, Dict[Any, str]] = collections.defaultdict(dict)
        local_index = {t: i for i, t in enumerate(topo_real)}
        task_begin = len(b.tasks)
        # a config change re-states tasks (e.g. AWS splits by zone while
        # reservations are configured)
        generation = (store.__dict__.get('_memo_generation', 0),
                      skypilot_config.generation())
        enabled_key = tuple(type(c) for c in enabled)
        for task in topo_real:
            slot_begin = b.n_slots
            res_list = list(task.resources)
            n_res = len(res_list)
            nodes = float(max(task.num_nodes, 0))
            num_nodes = task.num_nodes
            # A task stated before (same catalog, clouds, request objects,
            # node count) is replayed from its recorded slice of the problem:
            # its query / slot records are bytes that do not depend on the DAG
            # around it. Only the runtime (a user callback) is asked again.
            stated = task.__dict__.get('_stated')
            ids = tuple(map(id, res_list))
            if (stated is not None and stated[0] is store and
                    stated[1] == generation and stated[2] == enabled_key and
                    stated[3] is task.resources and stated[4] == ids and
                    stated[5] == (task.num_nodes > 1)):
                (q_recs, slot_recs, qbase_rel, slot_res, infos,
                 task_hints, free_slots) = stated[6]
                q0 = len(b.query_recs)
                b.query_recs.extend(q_recs)
                b.slot_recs.extend(slot_recs)
                b.slot_qbase.extend([q0 + r for r in qbase_rel])
                costs = []
                for res in res_list:
                    runtime = Optimizer._runtime(task, n_res, res)
                    costs.append((runtime / 3600, nodes, float(runtime)))
                flat = b.slot_cost
                if free_slots:
                    # on-premise clouds: the hourly cost is 0.0
                    for j, k in enumerate(slot_res):
                        flat.extend((0.0,) + costs[k][1:]
                                    if j in free_slots else costs[k])
                else:
                    for k in slot_res:
                        flat.extend(costs[k])
                slot_info.extend(infos)
                for res, by_cloud in task_hints.items():
                    hints[res].update(by_cloud)
            else:
                q_mark, info_mark = len(b.query_recs), len(slot_info)
                slot_res: List[int] = []
                free_slots = set()
                task_hints: Dict[Any, Dict[Any, str]] = {}
                for k, res in enumerate(res_list):
                    if res.__dict__.get('_validated_store') is not store:
                        # validate() is idempotent and only depends on the
                        # catalog
                        res.validate()
                        res.__dict__['_validated_store'] = store
                    if res.cloud is not None:
                        if not clouds.cloud_in_iterable(res.cloud, enabled):
                            continue
                        clouds_list = [res.cloud]
                    else:
                        clouds_list = enabled
                    runtime = float(Optimizer._runtime(task, n_res, res))
                    cost = (runtime / 3600, nodes, runtime)
                    free = (0.0, nodes, runtime)
                    for cloud in clouds_list:
                        table = tables.get(cloud.__class__, 0)
                        if table == 0:
                            name = cloud.canonical_name()
                            table = store.cloud(name) if store.has_cloud(
                                name) else None
                            tables[cloud.__class__] = table
                        if table is None:
                            continue
                        zero = table.rules.zero_cost
                        plan, slot = cloud.plan_cached(
                            b, res, num_nodes, free if zero else cost)
                        if plan.hint is not None:
                            hints[res][cloud] = plan.hint
                            task_hints.setdefault(res, {})[cloud] = plan.hint
                        if slot is None:
                            continue
                        if zero:
                            free_slots.add(len(slot_res))
                        slot_info.append(
                            _SlotInfo(task, res, cloud, plan, table))
                        slot_res.append(k)
                task.__dict__['_stated'] = (
                    store, generation, enabled_key, task.resources, ids,
                    task.num_nodes > 1,
                    (b.query_recs[q_mark:], b.slot_recs[slot_begin:],
                     [qb - q_mark for qb in b.slot_qbase[slot_begin:]],
                     slot_res, slot_info[info_mark:], task_hints,
                     free_slots))
            slot_end = b.n_slots
            parents = [
                p for p in dag_graph.predecessors(task) if not _is_dummy(p)
            ]
            edge_rows = []
            tariff_rows = store.__dict__.setdefault('_tariff_rows', {})
            for p in parents:
                nbytes = p.get_estimated_outputs_size_gigabytes()
                if not nbytes:
                    edge_rows.append([0.0] * n_clouds)
                elif minimize_cost:
                    # the clouds' piecewise tariffs are pure functions of the
                    # size: one row per distinct size
                    row = tariff_rows.get(nbytes)
                    if row is None:
                        row = [
                            float(c.get_egress_cost(num_gigabytes=nbytes))
                            for c in cloud_objs
                        ]
                        tariff_rows[nbytes] = row
                    edge_rows.append(row)
                else:
                    edge_rows.append([nbytes * 8 / 10] * n_clouds)
            src_row = None
            if not parents and task.get_inputs() is not None:
                nbytes = task.get_estimated_inputs_size_gigabytes()
                if nbytes:
                    src = task.get_inputs_cloud()
                    fn = (Optimizer._egress_cost
                          if minimize_cost else Optimizer._egress_time)
                    src_row = [float(fn(src, c, nbytes)) for c in cloud_objs]
            b.add_task(slot_begin, slot_end,
                       [local_index[p] for p in parents], edge_rows, src_row)
        blocked_begin = len(b.blocked)
        for blocked in blocked_resources or []:
            _add_blocked(b, store, blocked)
        b.add_dag(task_begin, len(b.tasks), is_chain, minimize_cost,
                  blocked_begin, len(b.blocked))
        return _Problem(b, list(topo_real), slot_info, hints, minimize_cost,
                        is_chain)

    @staticmethod
    def _solve(problem: _Problem, want_tables: bool = False) -> engine.Solution:
        problem.solution = engine.solve(problem.builder,
                                        device=catalog.get_device(),
                                        want_tables=want_tables)
        return problem.solution

    # ------------------------------------------------------------ _optimize_dag
    @staticmethod
    def _optimize_dag(
        dag: 'dag_lib.Dag',
        minimize_cost: bool = True,
        blocked_resources: Optional[Iterable[resources_lib.Resources]] = None,
        quiet: bool = False,
    ) -> Dict[task_lib.Task, resources_lib.Resources]:
        """Finds the optimal task -> Resources mapping for the whole DAG,
        egress included (sky/optimizer.py:1381-1512). `dag` carries the dummy
        source / sink like in the reference."""
        blocked = list(blocked_resources or [])
        ordered_choice = Optimizer._resolve_ordered_resources(dag, blocked)
        graph = dag.get_graph()
        topo_order = list(nx.topological_sort(graph))
        topo_real = [t for t in topo_order if not _is_dummy(t)]
        saved = {}
        for task, choice in ordered_choice.items():
            saved[task] = task.resources
            task.resources = {choice}
        try:
            problem = Optimizer._state_problem(graph, topo_real, minimize_cost,
                                               blocked, dag.is_chain())
            sol = Optimizer._solve(problem, want_tables=not quiet)
        finally:
            for task, original in saved.items():
                task.resources = original
        return Optimizer._apply_solution(problem, sol, graph, topo_order,
                                         topo_real, minimize_cost, blocked,
                                         quiet)

    @staticmethod
    def _apply_solution(problem, sol, graph, topo_order, topo_real,
                        minimize_cost, blocked, quiet):
        """Device result -> `best_resources` of every task (or the reference's
        ResourcesUnavailableError)."""
        res = sol.dag[0]
        if res['status'] == 1:
            failed = topo_real[int(res['task_fail'])]
            Optimizer._raise_unavailable(failed, blocked)
        if res['status'] != 0:
            # beyond the device enumeration: exact elimination on the host
            if sol.tables is None:
                sol = Optimizer._solve(problem, want_tables=True)
            _solve_large_dag(problem, sol, 0, 0, len(topo_real), minimize_cost)
            res = sol.dag[0]
        best_plan: Dict[task_lib.Task, resources_lib.Resources] = {}
        for i, task in enumerate(topo_real):
            launchable = problem.launchable(sol.chosen[i])
            task.best_resources = launchable
            best_plan[task] = launchable
        for t in topo_order:
            if _is_dummy(t):
                t.best_resources = list(t.resources)[0]
                best_plan[t] = t.best_resources
        if not quiet:
            objective = float(res['objective'])
            if minimize_cost:
                total_cost = objective
                total_time = Optimizer._compute_total_time(
                    graph, topo_order, best_plan)
            else:
                total_time = objective
                total_cost = Optimizer._compute_total_cost(
                    graph, topo_order, best_plan)
            Optimizer.print_optimized_plan(problem, sol, total_time,
                                           total_cost)
        return best_plan

    @staticmethod
    def session(dag: 'dag_lib.Dag',
                minimize: OptimizeTarget = OptimizeTarget.COST,
                quiet: bool = True) -> 'OptimizerSession':
        """Failover re-optimisation of one DAG: see OptimizerSession."""
        return OptimizerSession(dag, minimize, quiet)

    @staticmethod
    def _resolve_ordered_resources(dag, blocked) -> Dict[Any, Any]:
        """Ordered (list) resources: the first alternative with any launchable
        candidate wins; no joint optimisation (sky/optimizer.py:1403-1448).
        All alternatives of all such tasks are probed in one device call."""
        probes = []
        for task in dag.tasks:
            if isinstance(task.resources, list) and not _is_dummy(task):
                probes.append(task)
        if not probes:
            return {}
        store = catalog.get_store()
        b = engine.ProblemBuilder(store)
        graph = nx.DiGraph()
        index = []
        for task in probes:
            for alt in task.resources:
                probe = task_lib.Task.__new__(task_lib.Task)
                probe.__dict__.update(task.__dict__)
                probe.resources = {alt}
                graph.add_node(probe)
                Optimizer._state_problem(graph, [probe], True, blocked, True,
                                         builder=b)
                index.append((task, alt))
        sol = engine.solve(b, device=catalog.get_device())
        choice: Dict[Any, Any] = {}
        for i, (task, alt) in enumerate(index):
            if task not in choice and sol.task_n[i] > 0:
                choice[task] = alt
        for task in probes:
            # nothing launchable: keep the last alternative so that the error
            # message names a concrete request
            choice.setdefault(task, task.resources[-1])
        return choice

    # ------------------------------------------------ stand-alone DP / DAG search
    @staticmethod
    def _solve_cost_map(graph, topo_order, node_to_cost_map, minimize_cost,
                        is_chain):
        """Shared body of _optimize_by_dp / _optimize_by_ilp: the candidate
        tables of the reference's `node_to_cost_map` go to the device as they
        are (values in dictionary order + the candidate's cloud), the egress
        tariffs as per-edge scalars; the DP / exact search runs in
        solve_kernel (skyopt_solve_tables)."""
        store = catalog.get_store()
        cloud_objs = [_cloud_object(t.name) for t in store.clouds]
        n_clouds = len(cloud_objs)
        real = [t for t in topo_order if not _is_dummy(t)]
        index = {t: i for i, t in enumerate(real)}
        values, cl, parents, edge_rows, src_rows, keys = [], [], [], [], [], []
        for task in real:
            table = node_to_cost_map[task]
            keys.append(list(table.keys()))
            values.append([float(v) for v in table.values()])
            row = []
            for r in table.keys():
                name = r.cloud.canonical_name()
                if not store.has_cloud(name):
                    raise ValueError(f'{r.cloud} is not in the loaded catalog')
                row.append(store.cloud_index[name])
            cl.append(row)
            preds = [p for p in graph.predecessors(task) if not _is_dummy(p)]
            parents.append([index[p] for p in preds])
            rows = []
            for p in preds:
                nbytes = p.get_estimated_outputs_size_gigabytes()
                if not nbytes:
                    rows.append([0.0] * n_clouds)
                elif minimize_cost:
                    rows.append([float(c.get_egress_cost(num_gigabytes=nbytes))
                                 for c in cloud_objs])
                else:
                    rows.append([nbytes * 8 / 10] * n_clouds)
            edge_rows.append(rows)
            src = None
            if not preds and task.get_inputs() is not None:
                nbytes = task.get_estimated_inputs_size_gigabytes()
                if nbytes:
                    src_cloud = task.get_inputs_cloud()
                    fn = (Optimizer._egress_cost
                          if minimize_cost else Optimizer._egress_time)
                    src = [float(fn(src_cloud, c, nbytes)) for c in cloud_objs]
            src_rows.append(src)
        chosen, objective, status = engine.solve_tables(
            store, values, cl, parents, edge_rows, src_rows, is_chain,
            minimize_cost, device=catalog.get_device())
        if status == 2:
            # beyond the device enumeration (dag_solver.py)
            from skypilot_b200 import dag_solver  # pylint: disable=import-outside-toplevel
            if not minimize_cost:
                raise exceptions.OptimizerLimitError(
                    'The DAG is too large for the exact general-DAG search '
                    'under the TIME objective.')
            chosen, objective = dag_solver.solve_cost_dag(
                values, cl, parents, edge_rows, src_rows, n_clouds)
        elif status != 0:
            raise exceptions.ResourcesUnavailableError(
                'No launchable resource found for a task of the DAG.')
        best_plan = {}
        for task, idx, ks in zip(real, chosen, keys):
            task.best_resources = ks[idx]
            best_plan[task] = ks[idx]
        for t in topo_order:
            if _is_dummy(t):
                t.best_resources = list(t.resources)[0]
                best_plan[t] = t.best_resources
        return best_plan, objective

    @staticmethod
    def _optimize_by_dp(topo_order, node_to_cost_map, minimize_cost=True):
        """Chain DP on a given cost map (sky/optimizer.py:429-487)."""
        graph = nx.DiGraph()
        graph.add_nodes_from(topo_order)
        for a, b in zip(topo_order[:-1], topo_order[1:]):
            graph.add_edge(a, b)
        return Optimizer._solve_cost_map(graph, topo_order, node_to_cost_map,
                                         minimize_cost, True)

    @staticmethod
    def _optimize_by_ilp(graph, topo_order, node_to_cost_map,
                         minimize_cost=True):
        """General DAGs (sky/optimizer.py:490-637): the reference builds a
        0/1 ILP and calls CBC; here the exact optimum of the same objective
        comes from an exhaustive search on the device (DESIGN.md section 4)."""
        return Optimizer._solve_cost_map(graph, topo_order, node_to_cost_map,
                                         minimize_cost, False)

    # --------------------------------------------- object-level reference API
    @staticmethod
    def _estimate_nodes_cost_or_time(
        topo_order: List[task_lib.Task],
        minimize_cost: bool = True,
        blocked_resources: Optional[Iterable[resources_lib.Resources]] = None,
        quiet: bool = False
    ) -> Tuple[_TaskToCostMap, _TaskToPerCloudCandidates]:
        """node -> {launchable Resources -> cost or time}, in the reference's
        candidate order (sky/optimizer.py:239-426). The table is computed on
        the device; this wrapper only materialises the Resources objects."""
        del quiet
        node_to_cost_map: _TaskToCostMap = collections.defaultdict(dict)
        node_to_candidate_map: _TaskToPerCloudCandidates = {}
        real = [t for t in topo_order if not _is_dummy(t)]
        graph = nx.DiGraph()
        graph.add_nodes_from(real)
        problem = Optimizer._state_problem(graph, real, minimize_cost,
                                           list(blocked_resources or []), True)
        # every task is costed independently here: one single-task DAG each
        b = problem.builder
        b.dags = []
        n_blocked = len(b.blocked)
        for i in range(len(real)):
            b.set_task_field(i, 'n_parents', 0)
            b.add_dag(i, i + 1, True, minimize_cost, 0, n_blocked)
        sol = Optimizer._solve(problem, want_tables=True)
        for i, task in enumerate(real):
            if sol.task_n[i] == 0:
                Optimizer._raise_unavailable(task,
                                             list(blocked_resources or []))
            per_cloud: _PerCloudCandidates = collections.defaultdict(list)
            for cand in sol.task_table(i):
                launchable = problem.launchable(cand)
                value = float(cand['value'])
                node_to_cost_map[task][launchable] = value
                info = problem.slot_info[int(cand['slot'])]
                if not per_cloud[info.cloud]:
                    per_cloud[info.cloud].append(
                        info.plan.make(launchable.instance_type,
                                       info.resources))
            node_to_candidate_map[task] = per_cloud
        for t in topo_order:
            if _is_dummy(t):
                node_to_cost_map[t][list(t.resources)[0]] = 0
        return node_to_cost_map, node_to_candidate_map

    @staticmethod
    def _raise_unavailable(task, blocked) -> None:
        """Builds the reference's error text (sky/optimizer.py:368-425)."""
        _, _, fuzzy, resource_hints = _fill_in_launchable_resources(
            task, blocked, quiet=True)
        raise Optimizer._unavailable_error(task, fuzzy, resource_hints)

    @staticmethod
    def _unavailable_error(task, fuzzy, resource_hints
                          ) -> exceptions.ResourcesUnavailableError:
        fuzzy_str = ''
        if fuzzy:
            fuzzy_str = f'\nTry one of these offered accelerators: {fuzzy}'
        reprs = ', '.join(f'{task.num_nodes}x ' + r.repr_with_region_zone
                          for r in task.resources)
        indent = ' ' * len('Hint: ')
        hints_concat = '\n'.join(f'Resource: {r!r}\n' + '\n'.join(h)
                                 for r, h in resource_hints.items() if h)
        # like the reference: ''.split('\n') is [''], so without any hint the
        # text still ends in 'Hint: Check Per Resource Hint' and an indent
        hints_fmt = '\n'.join(
            f'{indent}{line}' for line in hints_concat.split('\n'))
        hints_str = (f'Hint: Check Per Resource Hint\n{hints_fmt}'
                     if hints_fmt else '')
        return exceptions.ResourcesUnavailableError(
            'Catalog does not contain any instances satisfying the request: '
            f'{reprs}.\nTo fix: relax or change the resource requirements.'
            f'{fuzzy_str}\n\nHint: sky gpus list to list available '
            f'accelerators.\n{indent}sky check to check the enabled clouds.\n'
            f'{hints_str}')

    @staticmethod
    def _unavailable_errors(tasks: List[task_lib.Task]
                           ) -> List[exceptions.ResourcesUnavailableError]:
        """The errors of many infeasible tasks from ONE device scan: every
        (request, cloud) of every task is stated into one batch with fuzzy
        candidates wanted (Cloud.feasible_begin); hints and fuzzy lists are
        collected exactly like `_fill_in_launchable_resources` does for one
        task. A batch with thousands of infeasible DAGs used to pay one
        scan per (task, cloud) just to word its errors."""
        enabled = sky_check.get_cached_enabled_clouds_or_refresh(
            raise_if_no_cloud_access=True)
        store = catalog.get_store()
        b = engine.ProblemBuilder(store)
        pending = []
        for task in tasks:
            per_task = []
            for resources in task.resources:
                resources.validate()
                if (resources.cloud is not None and
                        not clouds.cloud_in_iterable(resources.cloud,
                                                     enabled)):
                    continue
                clouds_list = ([resources.cloud]
                               if resources.cloud is not None else enabled)
                for cloud in clouds_list:
                    per_task.append(
                        (resources,
                         cloud.feasible_begin(b, resources, task.num_nodes)))
            pending.append(per_task)
        out = None
        if b.n_queries:
            out = engine.scan(b, fuzzy_cap=min(max(len(store.acc_keys), 1),
                                               2048),
                              device=catalog.get_device())
        errors = []
        for task, per_task in zip(tasks, pending):
            all_fuzzy = set()
            hints: Dict[Any, List[str]] = collections.defaultdict(list)
            for resources, end in per_task:
                feasible = end(out)
                if feasible.hint is not None:
                    hints[resources].append(feasible.hint)
                if not feasible.resources_list:
                    all_fuzzy.update(feasible.fuzzy_candidate_list)
            errors.append(
                Optimizer._unavailable_error(task, sorted(all_fuzzy), hints))
        return errors

    @staticmethod
    def _compute_total_time(graph, topo_order, plan) -> float:
        """Critical-path time of a plan (sky/optimizer.py:640-671)."""
        finish: Dict[Any, float] = {}

        def finish_time(node):
            if node in finish:
                return finish[node]
            resources = plan[node]
            if node.time_estimator_func is None:
                execution = 1 * 3600
            else:
                execution = node.estimate_runtime(resources)
            preds = [0]
            for pred in graph.predecessors(node):
                egress = Optimizer._egress_cost_or_time(False, pred,
                                                        plan[pred], node,
                                                        resources)
                preds.append(finish_time(pred) + egress)
            finish[node] = execution + max(preds)
            return finish[node]

        return finish_time(topo_order[-1])

    @staticmethod
    def _compute_total_cost(graph, topo_order, plan) -> float:
        """Execution + egress cost of a plan (sky/optimizer.py:674-698)."""
        total = 0.
        for node in topo_order:
            resources = plan[node]
            if node.time_estimator_func is None:
                execution = 1 * 3600
            else:
                execution = node.estimate_runtime(resources)
            total += resources.get_cost(execution) * node.num_nodes
            for pred in graph.predecessors(node):
                total += Optimizer._egress_cost_or_time(
                    True, pred, plan[pred], node, resources)
        return total

    @staticmethod
    def print_optimized_plan(problem: _Problem, sol: engine.Solution,
                             total_time: float, total_cost: float) -> None:
        """Logs the chosen plan and the per-task alternatives (compact form
        of sky/optimizer.py:738-1033)."""
        lines = []
        if len(problem.tasks) > 1:
            lines.append(f'Estimated total runtime: {total_time / 3600:.1f} '
                         f'hours; estimated total cost: ${total_cost:.1f}')
        for i, task in enumerate(problem.tasks):
            best = task.best_resources
            lines.append(
                f'{task}: {task.num_nodes}x {best.repr_with_region_zone} '
                f'${float(sol.chosen[i]["hourly"]):.4f}/hr '
                f'({int(sol.task_n[i])} candidates)')
        logger.info('Optimizer plan:\n  ' + '\n  '.join(lines))


class OptimizerSession:
    """`Optimizer.optimize(dag, blocked_resources=...)` for the provisioner's
    failover loop (sky/backends/cloud_vm_ray_backend.py:332-339, :1817-1825),
    where the same DAG is optimised again and again under a growing blocked
    list. The first `optimize()` is a full device solve; the expanded
    candidate sets stay on the device, and every later call only uploads the
    blocked wildcards and re-runs the blocked filter and the solver
    (`skyopt_session_resolve`). Results are those of `Optimizer.optimize`.

        with Optimizer.session(dag) as s:
            s.optimize()
            while launch_failed:
                blocked.append(failed_resources)
                s.optimize(blocked)

    Tasks with ordered (list) resources resolve their choice against the
    blocked list on the host first (optimizer.py:1403-1448), so they fall back
    to a full `Optimizer.optimize` per call.
    """

    def __init__(self, dag, minimize=OptimizeTarget.COST, quiet: bool = True):
        self.dag = dag
        self.minimize_cost = minimize == OptimizeTarget.COST
        self.minimize = minimize
        self.quiet = quiet
        self._session: Optional[engine.Session] = None
        self._problem = None
        # (reservation, config) generations the open session was stated under
        self._state_key = None
        self._fallback = any(isinstance(t.resources, list) for t in dag.tasks)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def close(self) -> None:
        if self._session is not None:
            self._session.close()
            self._session = None

    def optimize(self, blocked_resources=None):
        blocked = list(blocked_resources or [])
        if self._fallback:
            return Optimizer.optimize(self.dag, self.minimize, blocked,
                                      self.quiet)
        dag = self.dag
        _check_specified_clouds(dag)
        Optimizer._add_dummy_source_sink_nodes(dag)  # pylint: disable=protected-access
        try:
            graph = dag.get_graph()
            topo_order = list(nx.topological_sort(graph))
            topo_real = [t for t in topo_order if not _is_dummy(t)]
            store = catalog.get_store()
            if self._session is not None and store is not self._problem.builder.store:
                # region / zone / instance ids are ranks of ONE catalog: after
                # a reload the device-resident candidates mean something else
                raise RuntimeError(
                    'the catalog changed while an OptimizerSession was open; '
                    'close the session and open a new one')
            state_key = (reservations.generation(),
                         skypilot_config.generation())
            if self._session is not None and state_key != self._state_key:
                # new reservation counts or config: the device-resident
                # candidate values are stale, state the DAG again
                self.close()
            if self._session is None:
                self._state_key = state_key
                problem = Optimizer._state_problem(  # pylint: disable=protected-access
                    graph, topo_real, self.minimize_cost, blocked,
                    dag.is_chain())
                self._problem = problem
                if problem.builder.n_slots == 0:
                    sol = Optimizer._solve(problem)  # pylint: disable=protected-access
                else:
                    self._session = engine.Session(
                        problem.builder, device=catalog.get_device(),
                        want_tables=not self.quiet)
                    sol = self._session.solution
                    problem.solution = sol
            else:
                scratch = engine.ProblemBuilder(store)
                for r in blocked:
                    _add_blocked(scratch, store, r)
                sol = self._session.resolve(scratch.blocked)
                self._problem.solution = sol
            Optimizer._apply_solution(  # pylint: disable=protected-access
                self._problem, sol, graph, topo_order, topo_real,
                self.minimize_cost, blocked, self.quiet)
        finally:
            Optimizer._remove_dummy_source_sink_nodes(dag)  # pylint: disable=protected-access
        return dag


def _cloud_object(name: str) -> clouds.Cloud:
    from skypilot_b200.utils import registry  # pylint: disable=import-outside-toplevel
    if name in registry.CLOUD_REGISTRY:
        return registry.CLOUD_REGISTRY.from_str(name)
    return clouds.DummyCloud()


def _solve_large_dag(problem, sol, dag_index: int, task_begin: int,
                     n_tasks: int, minimize_cost: bool):
    """A general DAG the device enumeration refused (status 2: more than 16
    tasks or 2^26 cloud assignments): exact bucket elimination over the
    per-cloud minima of the candidate tables (dag_solver.py). Fills
    `sol.chosen` / `sol.dag` like the device does."""
    from skypilot_b200 import dag_solver  # pylint: disable=import-outside-toplevel
    if not minimize_cost:
        raise exceptions.OptimizerLimitError(
            'The DAG is too large for the exact general-DAG search under '
            'the TIME objective (more than 16 tasks or 2^26 cloud '
            'assignments); the COST objective has no such limit.')
    packed = sol.packed
    n_clouds = len(packed.store.clouds)
    values, cls, parents, edge_rows, src_rows = [], [], [], [], []
    for lt in range(n_tasks):
        t = task_begin + lt
        table = sol.task_table(t)
        values.append([float(v) for v in table['value']])
        cls.append([int(packed.slots['cloud'][int(sl)]) for sl in table['slot']])
        tk = packed.tasks[t]
        npar = int(tk['n_parents'])
        pb = int(tk['parent_begin'])
        parents.append([int(p) for p in packed.parents[pb:pb + npar]])
        eb = int(tk['edge_tariff_begin'])
        edge_rows.append([
            [float(x) for x in packed.tariffs[eb + j * n_clouds:
                                              eb + (j + 1) * n_clouds]]
            for j in range(npar)
        ])
        sb = int(tk['src_tariff_begin'])
        src_rows.append(None if (npar or sb < 0) else
                        [float(x) for x in packed.tariffs[sb:sb + n_clouds]])
    chosen, objective = dag_solver.solve_cost_dag(values, cls, parents,
                                                  edge_rows, src_rows, n_clouds)
    for lt, k in enumerate(chosen):
        t = task_begin + lt
        sol.chosen[t] = sol.task_table(t)[k]
        sol.chosen_index[t] = k
    sol.dag[dag_index]['status'] = 0
    sol.dag[dag_index]['task_fail'] = -1
    sol.dag[dag_index]['objective'] = objective


def _add_blocked(b: engine.ProblemBuilder, store, blocked) -> None:
    """One `should_be_blocked_by` wildcard (sky/resources.py:1938-1961) as
    device entries; names are resolved against each cloud's dictionaries."""
    targets = []
    if blocked.cloud is not None:
        name = blocked.cloud.canonical_name()
        if not store.has_cloud(name):
            return
        targets = [store.cloud(name)]
    else:
        targets = list(store.clouds)
    acc_key = -1
    accs = blocked.accelerators
    if accs is not None:
        if len(accs) != 1:
            return
        name, count = list(accs.items())[0]
        # -3: a name the catalog does not know matches no candidate -- not even
        # a candidate whose own accelerator is unknown (-2, clouds/gcp.py): the
        # reference compares the dicts themselves (sky/resources.py:1956-1958)
        acc_key = store.acc_key_index.get((name, float(count)), -3)
    needs_cloud = (blocked.instance_type is not None or
                   blocked.region is not None or blocked.zone is not None)
    if not needs_cloud and blocked.cloud is None:
        b.add_blocked(acc_key=acc_key, use_spot=int(blocked.use_spot))
        return
    for table in targets:
        entry = dict(cloud=table.index, acc_key=acc_key,
                     use_spot=int(blocked.use_spot))
        if blocked.instance_type is not None:
            entry['inst_id'] = table.inst_index.get(
                blocked.instance_type,
                -2 if blocked.instance_type != 'TPU-VM' else -2)
        if blocked.region is not None:
            entry['region_id'] = table.region_exact.get(blocked.region, -2)
        if blocked.zone is not None:
            entry['zone_id'] = table.zone_exact.get(blocked.zone, -2)
        b.add_blocked(**entry)


def _filter_out_blocked_launchable_resources(launchable_resources,
                                             blocked_resources):
    available = []
    for resources in launchable_resources:
        for blocked in blocked_resources:
            if resources.should_be_blocked_by(blocked):
                break
        else:
            available.append(resources)
    return available


def _check_specified_clouds(dag: 'dag_lib.Dag', enabled=None) -> None:
    """A task pinned to a cloud that is not enabled cannot be placed
    (sky/optimizer.py:1541-1607)."""
    if enabled is None:
        enabled = sky_check.get_cached_enabled_clouds_or_refresh(
            raise_if_no_cloud_access=True)
    for task in dag.tasks:
        specified, disabled = set(), set()
        for resources in task.resources:
            cloud_str = str(resources.cloud)
            if (resources.cloud is not None and
                    not clouds.cloud_in_iterable(resources.cloud, enabled)):
                disabled.add(cloud_str)
            specified.add(cloud_str)
        if disabled:
            is_or_are = 'is' if len(disabled) == 1 else 'are'
            task_name = f' {task.name!r}' if task.name is not None else ''
            msg = (f'Task{task_name} requires {", ".join(sorted(disabled))} '
                   f'which {is_or_are} not enabled. To enable access, change '
                   'the task cloud requirement or run: sky check '
                   f'{" ".join(c.lower() for c in sorted(disabled))}')
            if specified == disabled:
                raise exceptions.ResourcesUnavailableError(msg)
            logger.warning(msg)


def _fill_in_launchable_resources(
    task: task_lib.Task,
    blocked_resources: Optional[Iterable[resources_lib.Resources]],
    quiet: bool = False
) -> Tuple[Dict[resources_lib.Resources, List[resources_lib.Resources]],
           _PerCloudCandidates, List[str], Dict[resources_lib.Resources,
                                                List[str]]]:
    """requested Resources -> launchable Resources, per-cloud feasible lists,
    fuzzy candidates and hints (sky/optimizer.py:1664-1785). Object-level
    path: one `skyopt_scan` per cloud plus one expansion call per cheapest
    instance type."""
    enabled = sky_check.get_cached_enabled_clouds_or_refresh(
        raise_if_no_cloud_access=True)
    launchable: Dict[resources_lib.Resources,
                     List[resources_lib.Resources]] = (
                         collections.defaultdict(list))
    all_fuzzy = set()
    cloud_candidates: _PerCloudCandidates = collections.defaultdict(list)
    resource_hints: Dict[resources_lib.Resources,
                         List[str]] = collections.defaultdict(list)
    blocked = list(blocked_resources or [])
    for resources in task.resources:
        resources.validate()
        if (resources.cloud is not None and
                not clouds.cloud_in_iterable(resources.cloud, enabled)):
            launchable[resources] = []
            continue
        clouds_list = ([resources.cloud]
                       if resources.cloud is not None else enabled)
        for cloud in clouds_list:
            feasible = cloud.get_feasible_launchable_resources(
                resources, task.num_nodes)
            if feasible.hint is not None:
                resource_hints[resources].append(feasible.hint)
            if feasible.resources_list:
                cheapest = feasible.resources_list[0]
                launchable[resources].extend(
                    resources_utils.make_launchables_for_valid_region_zones(
                        cheapest))
                cloud_candidates[cloud].extend(feasible.resources_list)
            else:
                all_fuzzy.update(feasible.fuzzy_candidate_list)
        if not launchable[resources] and not (
                quiet or resources.no_missing_accel_warnings):
            logger.info(f'No resource satisfying '
                        f'{resources.repr_with_region_zone} on '
                        f'{clouds_list}.')
            if all_fuzzy:
                logger.info(f'Did you mean: {sorted(all_fuzzy)}')
        launchable[resources] = _filter_out_blocked_launchable_resources(
            launchable[resources], blocked)
    return launchable, cloud_candidates, sorted(all_fuzzy), resource_hints
