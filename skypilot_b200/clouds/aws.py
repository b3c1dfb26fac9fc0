"""Amazon Web Services (placement-relevant part of sky/clouds/aws.py)."""
from typing import Any, Dict, Optional

from skypilot_b200.clouds import cloud
from skypilot_b200.utils import registry
from skypilot_b200.utils import resources_utils


@registry.CLOUD_REGISTRY.register
class AWS(cloud.Cloud):
    """AWS: accelerators are part of the instance type; region-level
    on-demand candidates (zone-level with reservations configured), zone-level
    spot candidates (aws.py:347-371)."""
    _REPR = 'AWS'
    _CATALOG = 'aws'
    _DEFAULT_IMAGE_GB = 45  # DEFAULT_AMI_GB, sky/clouds/aws.py:59

    @classmethod
    def _unsupported_features_for_resources(cls, resources: Any,
                                            region: Optional[str] = None):
        # aws.py:302-324: stopping spot instances is the only dynamic entry
        # and it does not concern placement.
        del resources, region
        return {}

    @classmethod
    def optimize_by_zone(cls) -> bool:
        """One candidate per zone when reservations are configured
        (aws.py:369-371, aws_utils.use_reservations): reserved capacity is
        zonal, so on-demand candidates are priced zone by zone."""
        from skypilot_b200 import reservations  # pylint: disable=import-outside-toplevel
        return reservations.use_reservations('aws')

    def get_egress_cost(self, num_gigabytes: float) -> float:
        """Tiered $/GB out of AWS (aws.py:667-688)."""
        g = num_gigabytes
        if g > 150 * 1024:
            return 0.05 * g
        cost = 0.0
        if g >= 50 * 1024:
            cost += (g - 50 * 1024) * 0.07
            g -= 50 * 1024
        if g >= 10 * 1024:
            cost += (g - 10 * 1024) * 0.085
            g -= 10 * 1024
        if g > 1:
            cost += (g - 1) * 0.09
        cost += 0.0
        return cost

    def get_feasible_launchable_resources(
            self, resources: Any,
            num_nodes: int = 1) -> resources_utils.FeasibleResources:
        if resources.instance_type is not None:
            hint = self._feature_hint(resources, num_nodes)
            if hint is not None:
                return resources_utils.FeasibleResources([], [], hint)
            # aws.py:884-898: an explicit instance type must be offered in
            # the requested region / zone.
            regions = self.regions_with_offering(
                resources.instance_type, resources.accelerators,
                resources.use_spot, resources.region, resources.zone)
            if not regions:
                return resources_utils.FeasibleResources([], [], None)
            return resources_utils.FeasibleResources(
                [resources.copy(accelerators=None)], [], None)
        return super().get_feasible_launchable_resources(resources, num_nodes)

    def feasible_begin(self, b, resources: Any, num_nodes: int = 1):
        if resources.instance_type is not None:
            # the explicit-instance rule above is its own device call
            answer = self.get_feasible_launchable_resources(resources,
                                                            num_nodes)
            return lambda out: answer
        return super().feasible_begin(b, resources, num_nodes)
