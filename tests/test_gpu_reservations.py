"""Capacity reservations on the device vs the unmodified reference.

The `reservations` fixtures (tests/golden/reservations.json) were generated
by the reference with its cloud APIs answered from each scenario's snapshot
(oracle/ref_harness/run_reference_reservations.py). The device path must
return the same plan, the same ordered candidate tables with their values,
objective, total cost and total time -- in every kernel mode -- and sessions,
batches and a full-size chain with 10 000 reservations must agree with the
host's view.
"""
import os
import random
import subprocess
import sys

import networkx as nx
import pytest

import skypilot_b200 as sky
from skypilot_b200 import optimizer as opt_lib
from skypilot_b200 import reservations
from skypilot_b200 import skypilot_config
from skypilot_b200.reservations import Reservation
from tests import reservation_scenarios
from tests import scenario_runner as runner
from tests import scenarios

pytestmark = pytest.mark.gpu

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
Optimizer = opt_lib.Optimizer


def _records(scenario):
    return [Reservation(**r) for r in scenario['reservations']]


def _device_objective(scenario):
    """best_total_objective of the device solve (the scenario runner reports
    the plan's total cost, which ignores reservations like the reference's
    _compute_total_cost)."""
    minimize_cost = scenario.get('minimize', 'cost') == 'cost'
    dag, _ = runner.build_dag(scenario)
    graph = dag.get_graph()
    topo = list(nx.topological_sort(graph))
    problem = Optimizer._state_problem(graph, topo, minimize_cost,  # pylint: disable=protected-access
                                       runner.blocked_list(scenario),
                                       dag.is_chain())
    sol = Optimizer._solve(problem)  # pylint: disable=protected-access
    assert int(sol.dag[0]['status']) == 0
    return float(sol.dag[0]['objective'])


def run_reservation_scenario(scenario):
    reservations.set_reservations(_records(scenario))
    try:
        got = runner.run_scenario(scenario)
        if 'error' not in got:
            skypilot_config.set_config(scenario['config'])
            try:
                got['objective'] = _device_objective(scenario)
            finally:
                skypilot_config.set_config(None)
    finally:
        reservations.set_reservations(None)
    return got


def check_suite():
    """Every reservations scenario against its fixture: [(name, diffs)]."""
    payload = runner.load_golden('reservations')
    assert payload['catalog'] == reservation_scenarios.CATALOG
    golden = {r['name']: r for r in payload['records']}
    runner.activate_catalog(payload['catalog'])
    bad = []
    for sc in reservation_scenarios.reservation_scenarios():
        diffs = runner.compare(golden[sc['name']],
                               run_reservation_scenario(sc))
        if diffs:
            bad.append((sc['name'], diffs[:3]))
    return bad


@pytest.fixture(autouse=True)
def _clean_state():
    yield
    reservations.set_reservations(None)
    skypilot_config.set_config(None)


def _cases():
    return [pytest.param(sc, id=sc['name'])
            for sc in reservation_scenarios.reservation_scenarios()]


@pytest.mark.parametrize('scenario', _cases())
def test_reservation_scenario_matches_reference(scenario):
    payload = runner.load_golden('reservations')
    assert payload['catalog'] == reservation_scenarios.CATALOG
    golden = {r['name']: r for r in payload['records']}[scenario['name']]
    runner.activate_catalog(payload['catalog'])
    got = run_reservation_scenario(scenario)
    diffs = runner.compare(golden, got)
    assert not diffs, diffs


@pytest.mark.parametrize('mode,exp', [
    ('auto', None), ('fast-split', None), ('fast-noprune', None),
    ('queue', None), ('tile', None), ('stream', None),
    ('auto', '8'), ('auto', '16'),
])
def test_reservation_suite_in_every_kernel_mode(mode, exp):
    """The same fixtures through each kernel family: the fused step
    (place_body), its split and no-prune forms, and the round-1 kernels
    (gather_kernel). The knobs are read once per process: subprocesses."""
    code = ('import sys; sys.path.insert(0, ".")\n'
            'from tests import test_gpu_reservations as t\n'
            'bad = t.check_suite()\n'
            'assert not bad, bad\n'
            'print("reservations ok")\n')
    env = dict(os.environ)
    env.pop('SKYOPT_SCAN_MODE', None)
    env.pop('SKYOPT_EXP', None)
    if mode != 'auto':
        env['SKYOPT_SCAN_MODE'] = mode
    if exp is not None:
        env['SKYOPT_EXP'] = exp
    proc = subprocess.run([sys.executable, '-c', code], cwd=_ROOT, env=env,
                          capture_output=True, text=True, timeout=900,
                          check=False)
    assert proc.returncode == 0, proc.stdout[-3000:] + proc.stderr[-3000:]
    assert 'reservations ok' in proc.stdout


def _plan(dag):
    return [runner.res_record(t.best_resources) for t in dag.tasks]


def _by_name(name):
    return next(s for s in reservation_scenarios.reservation_scenarios()
                if s['name'] == name)


def test_session_follows_reservation_changes():
    runner.activate_catalog(reservation_scenarios.CATALOG)
    sc = _by_name('res_chain_nodes')
    skypilot_config.set_config(sc['config'])
    reservations.set_reservations(_records(sc))
    blocked = [sky.Resources(cloud=sky.clouds.AWS(), region='us-west-2',
                             zone='us-west-2a')]

    def fresh(blocked_list=None):
        dag, _ = runner.build_dag(sc)
        Optimizer.optimize(dag, blocked_resources=blocked_list, quiet=True)
        return _plan(dag)

    dag, _ = runner.build_dag(sc)
    with Optimizer.session(dag) as s:
        s.optimize()
        assert _plan(dag) == fresh()
        s.optimize(blocked)
        assert _plan(dag) == fresh(blocked)
        # the reserved p3.2xlarge capacity of us-west-2a is used up: the
        # next solve must see it
        before = _plan(dag)
        reservations.set_reservations(
            [r for r in _records(sc) if r.name != 'cr-open-p3'])
        s.optimize()
        assert _plan(dag) == fresh()
        assert _plan(dag) != before or before[0]['zone'] != 'us-west-2a'


def test_batch_equals_single_dags():
    runner.activate_catalog(reservation_scenarios.CATALOG)
    names = ['res_aws_open', 'res_nodes4', 'res_gcp_nodes2', 'res_spot',
             'res_chain_egress', 'res_diamond', 'res_blocked_gcp']
    config = _by_name('res_both_v100')['config']
    skypilot_config.set_config(config)
    reservations.set_reservations(_records(_by_name('res_both_v100')))
    dags = [runner.build_dag(_by_name(n))[0] for n in names]
    Optimizer.optimize_batch(dags)
    batch = [_plan(d) for d in dags]
    for name, got in zip(names, batch):
        dag, _ = runner.build_dag(_by_name(name))
        Optimizer.optimize(dag, quiet=True)
        assert _plan(dag) == got, name


def _host_objective(dag):
    """The COST objective of the returned plan recomputed on the host:
    cost_per_node * max(num_nodes - reserved, 0) per task plus egress."""
    graph = dag.get_graph()
    total = 0.0
    for task in dag.tasks:
        res = task.best_resources
        runtime = (3600 if task.time_estimator_func is None else
                   task.estimate_runtime(list(task.resources)[0]))
        reserved = sum(res.get_reservations_available_resources().values())
        total += res.get_cost(runtime) * max(task.num_nodes - reserved, 0)
        for parent in graph.predecessors(task):
            total += Optimizer._egress_cost_or_time(  # pylint: disable=protected-access
                True, parent, parent.best_resources, task, res)
    return total


def test_full_size_chain_with_ten_thousand_reservations():
    from skypilot_b200 import workloads  # pylint: disable=import-outside-toplevel
    store = runner.activate_catalog(scenarios.CATALOGS['cfg4_1m'])
    sc = workloads.chain_scenario(32)
    config = {'aws': {'prioritize_reservations': True},
              'gcp': {'prioritize_reservations': True}}
    skypilot_config.set_config(config)
    dag, _ = runner.build_dag(sc)
    Optimizer.optimize(dag, quiet=True)
    used = {(str(t.best_resources.cloud).lower(),
             t.best_resources.instance_type) for t in dag.tasks}
    rng = random.Random(20261017)
    records = []
    clouds = [c for c in ('aws', 'gcp') if store.has_cloud(c)]
    for i in range(10000):
        cloud = rng.choice(clouds)
        table = store.cloud(cloud)
        mine = [it for c, it in used if c == cloud]
        itype = (rng.choice(mine) if mine and rng.random() < 0.7 else
                 rng.choice(table.inst_names))
        zone = rng.choice(table.zone_names)
        region = table.region_names[table.zone_region[table.zone_exact[zone]]]
        records.append(Reservation(cloud, f'r-{i}', itype, region, zone,
                                   rng.randint(0, 3), rng.random() < 0.2))
    reservations.set_reservations(records)
    problem_dag, _ = runner.build_dag(sc)
    graph = problem_dag.get_graph()
    topo = list(nx.topological_sort(graph))
    problem = Optimizer._state_problem(graph, topo, True, [], True)  # pylint: disable=protected-access
    assert problem.builder.reservations[1] > 1000
    sol = Optimizer._solve(problem)  # pylint: disable=protected-access
    assert int(sol.dag[0]['status']) == 0
    device = float(sol.dag[0]['objective'])
    for i, task in enumerate(topo):
        task.best_resources = problem.launchable(sol.chosen[i])
    host = _host_objective(problem_dag)
    assert runner.close(device, host, rel=1e-9), (device, host)
    # and the public entry point picks the same plan
    dag2, _ = runner.build_dag(sc)
    Optimizer.optimize(dag2, quiet=True)
    assert _plan(dag2) == _plan(problem_dag)
