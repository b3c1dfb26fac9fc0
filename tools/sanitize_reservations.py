"""Workload for compute-sanitizer: the `reservations` fixture suite (reserved
capacity looked up by place_body / gather_kernel) in one kernel mode.

    compute-sanitizer --tool memcheck python tools/sanitize_reservations.py fast-split
"""
import sys
sys.path.insert(0, '.')
from tests import reservation_scenarios  # noqa: E402
from tests import scenario_runner as runner  # noqa: E402
from tests import test_gpu_reservations as suite  # noqa: E402

mode = sys.argv[1] if len(sys.argv) > 1 else 'auto'
store = runner.activate_catalog(reservation_scenarios.CATALOG)
store.set_scan_mode(mode)
bad = suite.check_suite()
print('mode', mode, 'mismatches', len(bad), bad[:2])
