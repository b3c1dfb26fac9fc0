"""The reference harness (run_reference.py) with active capacity reservations.

Test infrastructure only (build container only; see bootstrap.py). Same
command line and record format as run_reference.py; a scenario may carry a
`reservations` snapshot (tests/reservation_scenarios.py), and the
reference's cloud-API boundary answers from it: boto3's
`describe_capacity_reservations` and `gcloud compute reservations list`. The
reference's own gating (need_to_query_reservations, use_reservations) and
matching (zone, targeted / specificReservationRequired, selfLink names) run
unchanged.

usage: run_reference_reservations.py --catalog '{...}' --scenarios in.json
                                     --out out.json
"""
import contextlib
import json
import os
import re
import sys
from unittest import mock

_HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, _HERE)

import run_reference  # noqa: E402  pylint: disable=wrong-import-position


def _clear_reservation_caches():
    from sky.clouds.utils import aws_utils
    from sky.clouds.utils import gcp_utils
    for fn in (aws_utils.list_reservations_for_instance_type,
               gcp_utils._list_reservations_for_instance_type):  # pylint: disable=protected-access
        clear = getattr(fn, 'cache_clear', None)
        if clear is not None:
            clear()
        else:
            fn.cache.clear()


@contextlib.contextmanager
def _reservation_apis(records):
    """The reference's cloud-API boundary answered from a snapshot, so that
    its own gating and matching run (sky/clouds/utils/aws_utils.py:44-69,
    sky/clouds/utils/gcp_utils.py:130-175). A record is
    {cloud, name, instance_type, region, zone, available, targeted}."""
    from sky.adaptors import aws as aws_adaptor
    from sky.utils import subprocess_utils

    class _EC2:

        def __init__(self, region):
            self.region = region

        def describe_capacity_reservations(self, Filters):  # pylint: disable=invalid-name
            want = {f['Name']: f['Values'] for f in Filters}
            assert want.get('state') == ['active'], Filters
            out = []
            for r in records:
                if (r['cloud'] == 'aws' and r['region'] == self.region and
                        r['instance_type'] in want['instance-type']):
                    out.append({
                        'CapacityReservationId': r['name'],
                        'InstanceType': r['instance_type'],
                        'AvailabilityZone': r['zone'],
                        'AvailableInstanceCount': r['available'],
                        'InstanceMatchCriteria':
                            'targeted' if r.get('targeted') else 'open',
                    })
            return {'CapacityReservations': out}

    def client(service_name, **kwargs):
        assert service_name == 'ec2', service_name
        return _EC2(kwargs['region_name'])

    def run_with_retries(cmd, **kwargs):
        del kwargs
        m = re.search(r'machineType=(\S+) AND status=READY', cmd)
        assert cmd.startswith('gcloud compute reservations list') and m, cmd
        out = []
        for r in records:
            if r['cloud'] != 'gcp' or r['instance_type'] != m.group(1):
                continue
            # name projects/<p>/reservations/<r>, as derived from the selfLink
            # (gcp_utils.py:110-117)
            _, project, _, res_name = r['name'].split('/')
            zone_url = ('https://www.googleapis.com/compute/v1/projects/'
                        f'{project}/zones/{r["zone"]}')
            out.append({
                'selfLink': f'{zone_url}/reservations/{res_name}',
                'zone': zone_url,
                'specificReservation': {'count': r['available'] + 1,
                                        'inUseCount': 1},
                'specificReservationRequired': bool(r.get('targeted')),
            })
        return 0, json.dumps(out), ''

    _clear_reservation_caches()
    try:
        with mock.patch.object(aws_adaptor, 'client', client), \
                mock.patch.object(subprocess_utils, 'run_with_retries',
                                  run_with_retries):
            yield
    finally:
        _clear_reservation_caches()


_plain_run_scenario = run_reference.run_scenario


def run_scenario(sky, scenario):
    if scenario.get('reservations') is None:
        return _plain_run_scenario(sky, scenario)
    with _reservation_apis(scenario['reservations']):
        return _plain_run_scenario(sky, dict(scenario, reservations=None))


# run_reference.main() and its config wrapper call run_scenario by name
run_reference.run_scenario = run_scenario

if __name__ == '__main__':
    run_reference.main()
