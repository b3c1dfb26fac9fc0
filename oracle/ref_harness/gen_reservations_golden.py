"""Regenerate tests/golden/reservations.json from the UNMODIFIED reference.

Build container only (needs /root/reference). Runs the scenarios of
tests/reservation_scenarios.py through run_reference_reservations.py (the
reference harness with its cloud APIs answering from each scenario's
reservation snapshot) and writes the fixture in gen_golden.py's format:

    python oracle/ref_harness/gen_reservations_golden.py

The fixture is committed; the GPU box never runs this script.
"""
import json
import os
import subprocess
import sys
import tempfile

_HERE = os.path.dirname(os.path.abspath(__file__))
_REPO = os.path.dirname(os.path.dirname(_HERE))
sys.path.insert(0, _REPO)

from tests import reservation_scenarios  # noqa: E402  pylint: disable=wrong-import-position


def main():
    spec = dict(reservation_scenarios.CATALOG)
    suite = reservation_scenarios.reservation_scenarios()
    with tempfile.NamedTemporaryFile('w', suffix='.json', delete=False) as f:
        json.dump(suite, f)
        sc_path = f.name
    out_path = os.path.join(_REPO, 'tests', 'golden', 'reservations.json')
    tmp_out = out_path + '.tmp'
    cmd = [
        sys.executable,
        os.path.join(_HERE, 'run_reference_reservations.py'), '--catalog',
        json.dumps(spec), '--scenarios', sc_path, '--out', tmp_out
    ]
    print('[gen_reservations_golden]', len(suite), 'scenarios', flush=True)
    proc = subprocess.run(cmd, cwd='/tmp', stdout=subprocess.DEVNULL,
                          check=False)
    os.unlink(sc_path)
    if proc.returncode != 0:
        raise SystemExit('reference harness failed')
    with open(tmp_out, encoding='utf-8') as f:
        records = json.load(f)
    os.unlink(tmp_out)
    # compact candidates: [cloud, instance_type, region, zone, value]
    for rec in records:
        if 'candidates' in rec:
            rec['candidates'] = [[[
                c['cloud'], c['instance_type'], c['region'], c['zone'],
                c['value']
            ] for c in cands] for cands in rec['candidates']]
    payload = {
        'catalog': spec,
        'generated_by': 'oracle/ref_harness/gen_reservations_golden.py',
        'reference': 'skypilot-org/skypilot @ 7808630 (unmodified)',
        'records': records
    }
    with open(out_path, 'w', encoding='utf-8') as f:
        json.dump(payload, f, separators=(',', ':'), sort_keys=True)
    n_err = sum('error' in r for r in records)
    print(f'[gen_reservations_golden] wrote {out_path}: {len(records)} '
          f'records, {n_err} errors', flush=True)


if __name__ == '__main__':
    main()
