"""Capacity reservations on the host: the gating / consumability rule against
the reference's code (sky/resources.py:1785-1812, sky/clouds/aws.py:
1490-1519, sky/clouds/gcp.py:1419-1438, clouds/utils/*_utils.py), the device
table builder, the AWS per-zone statement and the extended C structs. No GPU.
"""
import ctypes

import pytest

import skypilot_b200 as sky
from skypilot_b200 import _native
from skypilot_b200 import engine
from skypilot_b200 import reservations
from skypilot_b200 import skypilot_config
from skypilot_b200 import synth
from skypilot_b200.reservations import Reservation
from tests import reservation_scenarios
from tests import scenario_runner as runner


@pytest.fixture(autouse=True)
def _clean_state():
    reservations.set_reservations(None)
    reservations.set_reservations_provider(None)
    skypilot_config.set_config(None)
    yield
    reservations.set_reservations(None)
    reservations.set_reservations_provider(None)
    skypilot_config.set_config(None)


@pytest.fixture(scope='module')
def store():
    return runner.activate_catalog(reservation_scenarios.CATALOG)


def _aws(name, zone, available, targeted=False, itype='p3.2xlarge',
         region=None):
    return Reservation('aws', name, itype, region or zone[:-1], zone,
                       available, targeted)


def _gcp(name, zone, available, targeted=False, itype='n1-highmem-8'):
    return Reservation('gcp', f'projects/p/reservations/{name}', itype,
                       zone.rsplit('-', 1)[0], zone, available, targeted)


def _cloud(name):
    from skypilot_b200.utils import registry  # pylint: disable=import-outside-toplevel
    return registry.CLOUD_REGISTRY.from_str(name)


def _launchable(store, cloud, itype, region, zone, use_spot=False):
    del store
    return sky.Resources(cloud=_cloud(cloud), instance_type=itype,
                         region=region, zone=zone, use_spot=use_spot)


# ------------------------------------------------------------------ the rule
def test_gate_needs_a_config(store):
    reservations.set_reservations([_aws('cr-1', 'us-west-2a', 2)])
    r = _launchable(store, 'aws', 'p3.2xlarge', 'us-west-2', 'us-west-2a')
    assert not reservations.need_to_query_reservations()
    assert r.get_reservations_available_resources() == {}
    skypilot_config.set_config({'aws': {'prioritize_reservations': True}})
    assert reservations.need_to_query_reservations()
    assert r.get_reservations_available_resources() == {'cr-1': 2}


def test_aws_consumability_and_summing(store):
    reservations.set_reservations([
        _aws('cr-open', 'us-west-2a', 2),
        _aws('cr-open-2', 'us-west-2a', 3),
        _aws('cr-tgt', 'us-west-2a', 5, targeted=True),
        _aws('cr-other-zone', 'us-west-2b', 7),
        _aws('cr-other-type', 'us-west-2a', 9, itype='m6i.2xlarge'),
    ])
    r = _launchable(store, 'aws', 'p3.2xlarge', 'us-west-2', 'us-west-2a')
    skypilot_config.set_config({'aws': {'prioritize_reservations': True}})
    assert r.get_reservations_available_resources() == {'cr-open': 2,
                                                        'cr-open-2': 3}
    # a targeted reservation counts once its id is listed
    skypilot_config.set_config({'aws': {'specific_reservations': ['cr-tgt']}})
    assert r.get_reservations_available_resources() == {
        'cr-open': 2, 'cr-open-2': 3, 'cr-tgt': 5}
    # an empty list is falsy: AWS does not consult its reservations
    skypilot_config.set_config({'aws': {'specific_reservations': []}})
    assert reservations.need_to_query_reservations()
    assert not reservations.use_reservations('aws')
    assert r.get_reservations_available_resources() == {}


def test_spot_zoneless_and_other_clouds(store):
    reservations.set_reservations([
        _aws('cr-open', 'us-west-2a', 2),
        Reservation('azure', 'az', 'Standard_D2s_v5', 'eastus', 'eastus-1',
                    3),
    ])
    skypilot_config.set_config({
        'aws': {'prioritize_reservations': True,
                'specific_reservations': ['cr-x']},
        'azure': {'prioritize_reservations': True}})
    spot = _launchable(store, 'aws', 'p3.2xlarge', 'us-west-2', 'us-west-2a',
                       use_spot=True)
    assert spot.get_reservations_available_resources() == {}
    # no zone: every listed reservation maps to 0 (aws.py:1498-1501)
    zoneless = _launchable(store, 'aws', 'p3.2xlarge', 'us-west-2', None)
    assert zoneless.get_reservations_available_resources() == {'cr-x': 0}
    azure = _launchable(store, 'azure', 'Standard_D2s_v5', 'eastus', None)
    assert azure.get_reservations_available_resources() == {}
    assert reservations.available_resources('azure', 'Standard_D2s_v5',
                                             'eastus', 'eastus-1',
                                             False) == {}


def test_gcp_rule(store):
    reservations.set_reservations([
        _gcp('open', 'us-west1-a', 1),
        _gcp('req', 'us-west1-a', 2, targeted=True),
        _gcp('other', 'us-west1-b', 4),
    ])
    r = _launchable(store, 'gcp', 'n1-highmem-8', 'us-west1', 'us-west1-a')
    skypilot_config.set_config({'gcp': {'prioritize_reservations': True}})
    assert r.get_reservations_available_resources() == {
        'projects/p/reservations/open': 1}
    skypilot_config.set_config(
        {'gcp': {'specific_reservations': ['projects/p/reservations/req']}})
    assert r.get_reservations_available_resources() == {
        'projects/p/reservations/open': 1, 'projects/p/reservations/req': 2}
    # only AWS' config is set: GCP's reservations are not consulted
    skypilot_config.set_config({'aws': {'prioritize_reservations': True}})
    assert r.get_reservations_available_resources() == {}


def test_provider_is_asked_per_gated_cloud(store):
    calls = []

    def provider(cloud):
        calls.append(cloud)
        return [_aws('cr-p', 'us-west-2a', 2)] if cloud == 'aws' else []

    reservations.set_reservations_provider(provider)
    skypilot_config.set_config({'aws': {'prioritize_reservations': True}})
    table, n = reservations.device_table(store)
    assert calls == ['aws'] and n == 1
    assert int(table['available'][0]) == 2


# ----------------------------------------------------------- table builder
def test_table_sorted_unique_and_mapped(store):
    recs = [
        _gcp('g1', 'us-west1-a', 1),
        _aws('cr-b', 'us-west-2b', 1),
        _aws('cr-a', 'us-west-2a', 2),
        _aws('cr-a2', 'us-west-2a', 3),
        _aws('cr-m', 'us-east-2b', 1, itype='m6i.2xlarge'),
        _aws('cr-zero', 'us-east-2a', 0, itype='m6i.2xlarge'),
        _aws('cr-unknown', 'us-east-1a', 5, itype='zz9.huge'),
        _aws('cr-badzone', 'us-east-1z', 5),
        _aws('cr-tgt', 'us-east-1a', 5, targeted=True),
    ]
    reservations.set_reservations(recs)
    skypilot_config.set_config({'aws': {'prioritize_reservations': True},
                                'gcp': {'prioritize_reservations': True}})
    table, n = reservations.device_table(store)
    rows = [tuple(int(x) for x in row) for row in table[:n]]
    assert rows == sorted(rows)
    assert len({r[:3] for r in rows}) == n
    aws, gcp = store.cloud('aws'), store.cloud('gcp')
    expect = {
        (aws.index, aws.inst_index['p3.2xlarge'], aws.zone_exact['us-west-2a']):
            5,
        (aws.index, aws.inst_index['p3.2xlarge'], aws.zone_exact['us-west-2b']):
            1,
        (aws.index, aws.inst_index['m6i.2xlarge'],
         aws.zone_exact['us-east-2b']): 1,
        (gcp.index, gcp.inst_index['n1-highmem-8'],
         gcp.zone_exact['us-west1-a']): 1,
    }
    assert {r[:3]: r[3] for r in rows} == expect
    # the memoised table follows the snapshot and the config
    skypilot_config.set_config({'gcp': {'prioritize_reservations': True}})
    _, n2 = reservations.device_table(store)
    assert n2 == 1
    skypilot_config.set_config(None)
    assert reservations.device_table(store)[1] == 0


@pytest.mark.parametrize('bad', [
    Reservation('aws', 'x', 'p3.2xlarge', 'us-west-2', 'us-west-2a', -1),
    Reservation('nosuchcloud', 'x', 'p3.2xlarge', 'r', 'z', 1),
    Reservation('aws', 'x', 'p3.2xlarge', 'us-west-2', None, 1),
    Reservation('aws', 'x', 'p3.2xlarge', 'us-west-2', '', 1),
    Reservation('aws', 'x', 'p3.2xlarge', 'us-west-2', 'us-west-2a', 1.5),
])
def test_malformed_records_raise(bad):
    before = reservations.generation()
    with pytest.raises(ValueError):
        reservations.set_reservations([bad])
    assert reservations.generation() == before


def test_duplicate_record_raises():
    rec = _aws('cr-1', 'us-west-2a', 1)
    with pytest.raises(ValueError):
        reservations.set_reservations([rec, rec])


def test_every_change_bumps_the_generation():
    g = reservations.generation()
    reservations.set_reservations([])
    reservations.set_reservations_provider(lambda cloud: [])
    reservations.set_reservations(None)
    assert reservations.generation() == g + 3


# ------------------------------------------------- AWS per-zone statement
def test_aws_slot_splits_by_zone_under_the_config(store):
    aws = sky.clouds.AWS()
    req = sky.Resources(cloud=aws, instance_type='p3.2xlarge')

    def split_flag():
        b = engine.ProblemBuilder(store)
        plan = aws.plan_feasible(b, req)
        assert plan.slot is not None
        packed = b.pack()
        return int(packed.slots['split_by_zone'][plan.slot])

    assert split_flag() == 0
    skypilot_config.set_config({'aws': {'prioritize_reservations': True}})
    assert aws.optimize_by_zone()
    assert split_flag() == 1
    skypilot_config.set_config(None)
    assert split_flag() == 0


# ------------------------------------------------------------ the C ABI
def test_extended_problem_layout():
    assert _native.ABI_VERSION == 4
    assert _native.RESERVATION_DTYPE.itemsize == 16
    assert list(_native.RESERVATION_DTYPE.names) == [
        'cloud', 'inst_id', 'zone_id', 'available']
    names = [f[0] for f in _native.Problem._fields_]
    assert names[-2:] == ['reservations', 'n_reservations']
    # appended at the end: every older field keeps its offset
    assert _native.Problem.dags.offset == 112
    assert _native.Problem.reservations.offset == 128
    assert ctypes.sizeof(_native.Problem) == 144
    assert _native.SLOT_DTYPE.itemsize == 80
    assert ctypes.sizeof(_native.Stats) == 56


def test_packed_problem_carries_the_table(store):
    reservations.set_reservations([_aws('cr-a', 'us-west-2a', 2)])
    skypilot_config.set_config({'aws': {'prioritize_reservations': True}})
    b = engine.ProblemBuilder(store)
    b.reservations = reservations.device_table(store)
    p = b.pack()
    assert p.n_reservations == 1
    c = p.c_problem()
    assert c.n_reservations == 1 and c.reservations
    empty = engine.ProblemBuilder(store).pack().c_problem()
    assert empty.n_reservations == 0 and not empty.reservations


# ---------------------------------------------- the fixture must bite
def test_reservation_fixture_changes_values():
    """In at least half of the COST records some candidate is valued below
    hourly * hours * num_nodes of its (instance type, zone) catalog rows."""
    payload = runner.load_golden('reservations')
    assert payload['catalog'] == reservation_scenarios.CATALOG
    frames = synth.make_catalogs(**payload['catalog'])
    cheapest = {}
    for cloud, df in frames.items():
        if 'AvailabilityZone' not in df:
            continue
        g = df.dropna(subset=['InstanceType', 'Price']).groupby(
            ['InstanceType', 'AvailabilityZone'])['Price'].min()
        for (itype, zone), price in g.items():
            cheapest[(cloud, itype, zone)] = float(price)
    by_name = {s['name']: s for s in reservation_scenarios.reservation_scenarios()}
    cost_records = bitten = 0
    for rec in payload['records']:
        sc = by_name[rec['name']]
        if sc.get('minimize', 'cost') != 'cost' or 'candidates' not in rec:
            continue
        cost_records += 1
        hit = False
        for task, cands in zip(sc['tasks'], rec['candidates']):
            nodes = task.get('num_nodes', 1)
            for cloud, itype, _, zone, value in cands:
                floor = cheapest.get((cloud, itype, zone))
                if floor is not None and value < floor * nodes * (1 - 1e-9):
                    hit = True
        bitten += hit
    assert cost_records >= 20
    assert bitten * 2 >= cost_records, (bitten, cost_records)
