"""Cost of the reservation look-up on the cfg4 chain (32 tasks, 1M-row
catalog): device step time (skyopt_optimize_timed, L2 flushed) and
end-to-end Optimizer.optimize p50 under three settings -- no config; the
reservation config with an empty snapshot; the config with 10 000 seeded
reservations (70% on the instance types of the unreserved plan). Prints one
JSON line per setting and one with the card's name and power limit.

    python tools/bench_reservations.py [--iters 200] [--e2e 30]
"""
import argparse
import json
import random
import statistics
import subprocess
import sys
import time

import networkx as nx

sys.path.insert(0, '.')
import skypilot_b200 as sky  # noqa: E402
from skypilot_b200 import engine  # noqa: E402
from skypilot_b200 import reservations  # noqa: E402
from skypilot_b200 import skypilot_config  # noqa: E402
from skypilot_b200 import synth  # noqa: E402
from skypilot_b200 import workloads  # noqa: E402
from skypilot_b200.reservations import Reservation  # noqa: E402
from tests import scenario_runner as runner  # noqa: E402

CONFIG = {'aws': {'prioritize_reservations': True},
          'gcp': {'prioritize_reservations': True}}


def seeded_reservations(store, used, n, seed=20261017):
    rng = random.Random(seed)
    clouds = [c for c in ('aws', 'gcp') if store.has_cloud(c)]
    out = []
    for i in range(n):
        cloud = rng.choice(clouds)
        table = store.cloud(cloud)
        mine = [it for c, it in used if c == cloud]
        itype = (rng.choice(mine) if mine and rng.random() < 0.7 else
                 rng.choice(table.inst_names))
        zone = rng.choice(table.zone_names)
        region = table.region_names[table.zone_region[table.zone_exact[zone]]]
        out.append(Reservation(cloud, f'r-{i}', itype, region, zone,
                               rng.randint(1, 3), rng.random() < 0.2))
    return out


def measure(scenario, iters, e2e):
    dag, _ = runner.build_dag(scenario)
    graph = dag.get_graph()
    topo = list(nx.topological_sort(graph))
    problem = sky.Optimizer._state_problem(graph, topo, True, [], True)  # pylint: disable=protected-access
    n_res = problem.builder.reservations[1]
    engine.solve_timed(problem.builder, 20)  # warm-up
    sol, iter_ms, _ = engine.solve_timed(problem.builder, iters)
    times = []
    for _ in range(e2e + 3):
        d, _ = runner.build_dag(scenario)
        t0 = time.perf_counter()
        sky.Optimizer.optimize(d, quiet=True)
        times.append(time.perf_counter() - t0)
    return {
        'n_reservation_entries': int(n_res),
        'step_p50_ms': float(statistics.median(iter_ms)),
        'step_min_ms': float(min(iter_ms)),
        'e2e_p50_ms': 1e3 * statistics.median(times[3:]),
        'objective': float(sol.dag[0]['objective']),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=200)
    ap.add_argument('--e2e', type=int, default=30)
    ap.add_argument('--n', type=int, default=10000)
    args = ap.parse_args()
    w = workloads.WORKLOADS['cfg4']
    sky.catalog.load_frames(synth.make_catalogs(**w['catalog']))
    store = sky.catalog.get_store()
    sky.check.set_enabled_clouds(sky.check.ALL_CATALOG_CLOUDS)
    scenario = workloads.chain_scenario(w['tasks'])
    try:
        gpu = subprocess.run(
            ['nvidia-smi', '--query-gpu=name,power.limit',
             '--format=csv,noheader'], capture_output=True, text=True,
            check=False).stdout.strip()
    except OSError:
        gpu = 'unknown'
    print(json.dumps({'gpu': gpu}), flush=True)
    print(json.dumps(dict(setting='no_config',
                          **measure(scenario, args.iters, args.e2e))),
          flush=True)
    skypilot_config.set_config(CONFIG)
    reservations.set_reservations([])
    print(json.dumps(dict(setting='config_empty_snapshot',
                          **measure(scenario, args.iters, args.e2e))),
          flush=True)
    dag, _ = runner.build_dag(scenario)
    sky.Optimizer.optimize(dag, quiet=True)
    used = {(str(t.best_resources.cloud).lower(),
             t.best_resources.instance_type) for t in dag.tasks}
    reservations.set_reservations(seeded_reservations(store, used, args.n))
    print(json.dumps(dict(setting=f'config_{args.n}_reservations',
                          **measure(scenario, args.iters, args.e2e))),
          flush=True)
    reservations.set_reservations(None)
    skypilot_config.set_config(None)


if __name__ == '__main__':
    main()
