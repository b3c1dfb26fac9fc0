"""`Resources`: a request for / a description of a launchable offering.

The placement-relevant surface of sky/resources.py: the constraint fields
(:148-440), `validate` (:442-456), `get_cost` (:1685-1698),
`get_valid_regions_for_launchable` (:1193-1246), `should_be_blocked_by`
(:1938-1961), `get_required_cloud_features` (:2156-2183) and `copy`
(:2076-2143). Like the reference there is no `__eq__` / `__hash__`:
Resources are identity-hashed dictionary keys.
"""
import re
from typing import Any, Dict, List, Optional, Set, Tuple, Union

from skypilot_b200 import check as sky_check
from skypilot_b200 import clouds
from skypilot_b200 import exceptions
from skypilot_b200.utils import registry
from skypilot_b200.utils import resources_utils

DEFAULT_DISK_SIZE_GB = 256


def canonicalize_accelerator_name(accelerator: str,
                                  cloud: Optional[clouds.Cloud]) -> str:
    """Catalog spelling of an accelerator name ('a100' -> 'A100'), following
    sky/utils/accelerator_registry.py:84-132 with the loaded catalog's
    accelerator dictionary in place of common/accelerators.csv."""
    if accelerator.lower().startswith('tpu-'):
        return accelerator.lower()
    from skypilot_b200 import catalog  # pylint: disable=import-outside-toplevel
    store = catalog.get_store(required=False)
    if store is None:
        return accelerator
    cloud_name = None if cloud is None else cloud.canonical_name()
    memo = store.__dict__.setdefault('_canonical_acc_names', {})
    hit = memo.get((accelerator, cloud_name))
    if hit is not None:
        return hit
    memo[(accelerator, cloud_name)] = name = _canonical_name(
        store, accelerator, cloud_name)
    return name


def _canonical_name(store, accelerator: str, cloud_name: Optional[str]) -> str:
    pattern = re.compile(accelerator, flags=re.IGNORECASE)
    by_name = store.accelerator_name_clouds()
    names = []
    for name, where in sorted(by_name.items()):
        if pattern.search(name) is None:
            continue
        if accelerator.lower() == name.lower():
            return name
        if cloud_name is None or cloud_name in where:
            names.append(name)
    if not names:
        return accelerator
    if len(names) == 1:
        return names[0]
    raise ValueError(f'Accelerator name {accelerator!r} is ambiguous. '
                     f'Please choose one of {names}.')


class Resources:
    """A (possibly partial) resource request; launchable once a cloud and an
    instance type are fixed."""

    def __init__(
        self,
        cloud: Optional[clouds.Cloud] = None,
        instance_type: Optional[str] = None,
        cpus: Union[None, int, float, str] = None,
        memory: Union[None, int, float, str] = None,
        accelerators: Union[None, str, Dict[str, Union[int, float]]] = None,
        accelerator_args: Optional[Dict[str, Any]] = None,
        infra: Optional[str] = None,
        use_spot: Optional[bool] = None,
        job_recovery: Optional[Union[Dict[str, Any], str]] = None,
        region: Optional[str] = None,
        zone: Optional[str] = None,
        image_id: Union[Dict[Optional[str], str], str, None] = None,
        disk_size: Optional[Union[str, int]] = None,
        disk_tier: Optional[Union[str, resources_utils.DiskTier]] = None,
        network_tier: Optional[Union[str,
                                     resources_utils.NetworkTier]] = None,
        local_disk: Optional[str] = None,
        max_hourly_cost: Optional[float] = None,
        ports: Optional[Union[int, str, List[str], Tuple[str]]] = None,
        labels: Optional[Dict[str, str]] = None,
        _no_missing_accel_warnings: Optional[bool] = None,
    ):
        if infra is not None:
            if cloud is not None or region is not None or zone is not None:
                raise ValueError(
                    'Cannot specify both `infra` and `cloud`, `region`, or '
                    f'`zone` parameters. Got: infra={infra}, cloud={cloud}, '
                    f'region={region}, zone={zone}')
            parts = [p for p in infra.strip('/').split('/')]
            cloud = registry.CLOUD_REGISTRY.from_str(
                parts[0]) if parts[0] not in ('', '*') else None
            region = parts[1] if len(parts) > 1 and parts[1] != '*' else None
            zone = parts[2] if len(parts) > 2 and parts[2] != '*' else None
        self._cloud = cloud
        self._region: Optional[str] = region
        self._zone: Optional[str] = zone
        self._instance_type = instance_type
        self._use_spot_specified = use_spot is not None
        self._use_spot = use_spot if use_spot is not None else False
        if isinstance(job_recovery, str):
            job_recovery = {'strategy': job_recovery}
        self._job_recovery = job_recovery
        if disk_size is not None:
            self._disk_size = int(
                resources_utils.parse_memory_resource(disk_size, 'disk_size'))
        else:
            self._disk_size = DEFAULT_DISK_SIZE_GB
        if isinstance(image_id, str):
            self._image_id: Optional[Dict[Optional[str], str]] = {
                self._region: image_id.strip()
            }
        elif isinstance(image_id, dict):
            if None in image_id:
                self._image_id = {self._region: image_id[None].strip()}
            else:
                self._image_id = {
                    k.strip(): v.strip() for k, v in image_id.items()
                }
        else:
            self._image_id = image_id
        if isinstance(disk_tier, str):
            tier = disk_tier.lower()
            supported = [t.value for t in resources_utils.DiskTier]
            if tier not in supported:
                raise ValueError(f'Invalid disk_tier {tier!r}. Disk tier must '
                                 f'be one of {", ".join(supported)}.')
            disk_tier = resources_utils.DiskTier(tier)
        self._disk_tier = disk_tier
        if isinstance(network_tier, str):
            tier = network_tier.lower()
            supported = [t.value for t in resources_utils.NetworkTier]
            if tier not in supported:
                raise ValueError(f'Invalid network_tier {tier!r}. Network tier '
                                 f'must be one of {", ".join(supported)}.')
            network_tier = resources_utils.NetworkTier(tier)
        self._network_tier = network_tier
        if ports is not None:
            if isinstance(ports, tuple):
                ports = list(ports)
            if not isinstance(ports, list):
                ports = [str(ports)]
            ports = [str(p) for p in ports] or None
        self._ports = ports
        self._labels = labels
        self._no_missing_accel_warnings = _no_missing_accel_warnings
        self._set_cpus(cpus)
        self._set_memory(memory)
        self._set_accelerators(accelerators, accelerator_args)
        self._local_disk = (None if local_disk is None else
                            resources_utils.normalize_local_disk(local_disk))
        self._max_hourly_cost = max_hourly_cost
        if self._image_id is not None:
            self._try_validate_image_id()

    def _try_validate_image_id(self) -> None:
        """The checks of Resources._try_validate_image_id that need no cloud
        API (sky/resources.py:1384-1500): docker images and custom images as
        features of the cloud, the image of a pinned region, `skypilot:` tags
        against <cloud>/images.csv, the stock image against disk_size."""
        f = clouds.CloudImplementationFeatures
        if self.extract_docker_image() is not None:
            if self._cloud is not None:
                self._cloud.check_features_are_supported(self,
                                                         {f.DOCKER_IMAGE})
            return
        if self._cloud is None:
            raise ValueError(
                'Cloud must be specified when image_id is provided.')
        try:
            self._cloud.check_features_are_supported(self, {f.IMAGE_ID})
        except exceptions.NotSupportedError as e:
            if self._cloud.is_same_cloud(clouds.Lambda()):
                raise ValueError(
                    'Lambda cloud only supports Docker images. '
                    'Please prefix your image with "docker:" '
                    '(e.g., image_id: docker:your-image-name).') from e
            raise ValueError(
                'image_id is only supported for AWS/GCP/Azure/IBM/OCI/'
                'Kubernetes/Nebius. For Lambda cloud, use "docker:" '
                'prefix for Docker images.') from e
        if self._region is not None:
            if None in self._image_id:
                self._image_id = {self._region: self._image_id[None]}
            elif self._region not in self._image_id:
                raise ValueError(
                    f'image_id {self._image_id} should contain the image '
                    f'for the specified region {self._region}.')
            else:
                self._image_id = {self._region: self._image_id[self._region]}
        for region, image_id in self._image_id.items():
            if (image_id.startswith('skypilot:') and
                    not self._cloud.is_image_tag_valid(image_id, region)):
                region_str = f' ({region})' if region else ''
                raise ValueError(
                    f'Image tag {image_id!r} is not valid, please make sure'
                    f' the tag exists in {self._cloud}{region_str}.')
            if (self._cloud.is_same_cloud(clouds.AWS()) and
                    not image_id.startswith('skypilot:') and region is None):
                raise ValueError(
                    'image_id is only supported for AWS in a specific '
                    'region, please explicitly specify the region.')
        for region, image_id in self._image_id.items():
            image_size = self._cloud.get_image_size(image_id, region)
            if image_size > self.disk_size:
                raise ValueError(
                    f'Image {image_id!r} is {image_size}GB, which is '
                    f'larger than the specified disk_size: {self.disk_size}'
                    ' GB. Please specify a larger disk_size to use this '
                    'image.')

    # ---- setters ------------------------------------------------------------
    def _set_cpus(self, cpus) -> None:
        if cpus is None:
            self._cpus = None
            return
        self._cpus = str(cpus)
        text = self._cpus
        body = text[:-1] if text.endswith('+') else text
        try:
            number = float(body)
        except ValueError:
            raise ValueError('The "cpus" field should be either a number or '
                             f'a string "<number>+". Found: {cpus!r}') from None
        if number <= 0:
            raise ValueError(
                f'The "cpus" field should be positive. Found: {cpus!r}')

    def _set_memory(self, memory) -> None:
        if memory is None:
            self._memory = None
            return
        text = resources_utils.parse_memory_resource(str(memory), 'memory',
                                                     ret_type=float,
                                                     allow_plus=True,
                                                     allow_x=True)
        self._memory = text
        body = text[:-1] if text.endswith(('+', 'x')) else text
        try:
            number = float(body)
        except ValueError:
            raise ValueError(
                'The "memory" field should be either a number or a string '
                f'"<number>+". Found: {memory!r}') from None
        if number <= 0:
            raise ValueError(
                f'The "memory" field should be positive. Found: {memory!r}')

    def _set_accelerators(self, accelerators, accelerator_args) -> None:
        if accelerators is not None:
            if isinstance(accelerators, str):
                if ':' not in accelerators:
                    accelerators = {accelerators: 1}
                else:
                    parts = accelerators.split(':')
                    error = ('The "accelerators" field as a str should be '
                             f'<name> or <name>:<cnt>. Found: {accelerators!r}')
                    if len(parts) != 2:
                        raise ValueError(error)
                    try:
                        num = float(parts[1])
                    except ValueError:
                        raise ValueError(error) from None
                    accelerators = {
                        parts[0]: int(num) if num.is_integer() else num
                    }
            acc = list(accelerators.keys())[0]
            if 'tpu' in acc.lower():
                # TPUs exist on GCP only in this catalog
                # (sky/resources.py:887-935).
                if self._cloud is None:
                    self._cloud = clouds.GCP()
                assert self._cloud.is_same_cloud(clouds.GCP()), (
                    'Cloud must be GCP for TPU accelerators.')
                if accelerator_args is None:
                    accelerator_args = {}
                use_tpu_vm = accelerator_args.get('tpu_vm', True)
                if 'runtime_version' not in accelerator_args:
                    if not use_tpu_vm:
                        version = '2.12.0'
                    elif acc.startswith('tpu-v5'):
                        version = 'v2-alpha-tpuv5'
                    elif acc.startswith('tpu-v6e'):
                        version = 'v2-alpha-tpuv6e'
                    else:
                        version = 'tpu-vm-base'
                    accelerator_args['runtime_version'] = version
                if (self._instance_type is not None and use_tpu_vm and
                        self._instance_type != 'TPU-VM'):
                    raise ValueError('Cannot specify instance type (got '
                                     f'{self._instance_type!r}) for TPU VM.')
        self._accelerators = accelerators
        self._accelerator_args = accelerator_args

    # ---- properties -----------------------------------------------------------
    @property
    def cloud(self) -> Optional[clouds.Cloud]:
        return self._cloud

    @property
    def region(self) -> Optional[str]:
        return self._region

    @property
    def zone(self) -> Optional[str]:
        return self._zone

    @property
    def instance_type(self) -> Optional[str]:
        return self._instance_type

    @property
    def cpus(self) -> Optional[str]:
        if self._cpus is not None:
            return self._cpus
        if self._cloud is not None and self._instance_type is not None:
            vcpus, _ = self._cloud.get_vcpus_mem_from_instance_type(
                self._instance_type)
            if vcpus is not None:
                return str(vcpus)
        return None

    @property
    def memory(self) -> Optional[str]:
        if self._memory is not None:
            return self._memory
        if self._cloud is not None and self._instance_type is not None:
            _, mem = self._cloud.get_vcpus_mem_from_instance_type(
                self._instance_type)
            if mem is not None:
                return str(mem)
        return None

    @property
    def accelerators(self) -> Optional[Dict[str, Union[int, float]]]:
        """Explicit accelerators, or the ones implied by the instance type."""
        if self._accelerators is not None:
            return self._accelerators
        if self._cloud is not None and self._instance_type is not None:
            return self._cloud.get_accelerators_from_instance_type(
                self._instance_type)
        return None

    @property
    def accelerator_args(self) -> Optional[Dict[str, Any]]:
        return self._accelerator_args

    @property
    def use_spot(self) -> bool:
        return self._use_spot

    @property
    def use_spot_specified(self) -> bool:
        return self._use_spot_specified

    @property
    def job_recovery(self):
        return self._job_recovery

    @property
    def disk_size(self) -> int:
        return self._disk_size

    @property
    def image_id(self) -> Optional[Dict[Optional[str], str]]:
        return self._image_id

    @property
    def disk_tier(self) -> Optional[resources_utils.DiskTier]:
        return self._disk_tier

    @property
    def network_tier(self) -> Optional[resources_utils.NetworkTier]:
        return self._network_tier

    @property
    def local_disk(self) -> Optional[str]:
        return self._local_disk

    @property
    def max_hourly_cost(self) -> Optional[float]:
        return self._max_hourly_cost

    @property
    def ports(self) -> Optional[List[str]]:
        return self._ports

    @property
    def labels(self) -> Optional[Dict[str, str]]:
        return self._labels

    @property
    def no_missing_accel_warnings(self) -> bool:
        return bool(self._no_missing_accel_warnings)

    # ---- representation ------------------------------------------------------
    def get_accelerators_str(self) -> str:
        accs = self.accelerators
        if accs is None:
            return ''
        return ', '.join(f'{k}:{v}' for k, v in accs.items())

    def get_spot_str(self) -> str:
        return '[Spot]' if self.use_spot else ''

    def __repr__(self) -> str:
        """The reference's text (sky/resources.py:448-568): it is part of the
        optimizer's error messages and tables. `<Cloud>(...)` without a cloud;
        inside the parentheses instance type[Spot], cpus, mem, accelerators,
        accelerator_args, image_id, disk_tier, network_tier, disk_size,
        local_disk, max_cost, ports -- the fields that are set."""
        fields = []
        if self.accelerators is not None:
            fields.append(f'{self.accelerators}')
            if self.accelerator_args is not None:
                fields.append(f'accelerator_args={self.accelerator_args}')
        head = []
        if self._cpus is not None:
            head.append(f'cpus={self._cpus}')
        if self.memory is not None:
            head.append(f'mem={self.memory}')
        tail = []
        if self.image_id is not None:
            tail.append(f'image_id={self.image_id[None]}' if None in
                        self.image_id else f'image_id={self.image_id}')
        if self.disk_tier is not None:
            tail.append(f'disk_tier={self.disk_tier.value}')
        if self.network_tier is not None:
            tail.append(f'network_tier={self.network_tier.value}')
        if self.disk_size != DEFAULT_DISK_SIZE_GB:
            tail.append(f'disk_size={self.disk_size}')
        if self._local_disk is not None:
            tail.append(f'local_disk={self._local_disk}')
        if self._max_hourly_cost is not None:
            tail.append(f'max_cost=${self._max_hourly_cost}/hr')
        if self.ports is not None:
            tail.append(f'ports={self.ports}')
        first = (self._instance_type or '') + ('[Spot]' if self.use_spot
                                                else '')
        parts = ([first] if first else []) + head + fields + tail
        cloud = '<Cloud>' if self._cloud is None else f'{self._cloud}'
        return f'{cloud}({", ".join(parts)})'

    @property
    def repr_with_region_zone(self) -> str:
        """sky/resources.py:571-586."""
        where = ''
        if self._region is not None:
            name = self._region
            if name.startswith('ssh-'):
                name = name[len('ssh-'):]
            where += f', region={name}'
        if self._zone is not None:
            where += f', zone={self._zone}'
        text = str(self)
        if text.endswith(')'):
            return text[:-1] + where + ')'
        return text + where

    # ---- validation -----------------------------------------------------------
    def validate(self) -> None:
        """Checks the request against the catalog and fills what can be
        inferred (canonical accelerator name, the zone's region, the cloud of
        an instance type): sky/resources.py:442-456."""
        self._try_canonicalize_accelerators()
        self._try_validate_and_set_region_zone()
        self._try_validate_instance_type()
        self._try_validate_cpus_mem()
        self._try_validate_misc()

    def _try_canonicalize_accelerators(self) -> None:
        if self._accelerators is None:
            return
        self._accelerators = {
            canonicalize_accelerator_name(acc, self._cloud): count
            for acc, count in self._accelerators.items()
        }

    def _try_validate_and_set_region_zone(self) -> None:
        if self._region is None and self._zone is None:
            return
        if self._cloud is None:
            enabled = sky_check.get_cached_enabled_clouds_or_refresh(
                raise_if_no_cloud_access=True)
            valid, errors = [], {}
            for cloud in enabled:
                try:
                    cloud.validate_region_zone(self._region, self._zone)
                except ValueError as e:
                    errors[repr(cloud)] = e
                    continue
                valid.append(cloud)
            if not valid:
                where = (f'for cloud {enabled[0]}' if len(enabled) == 1 else
                         f'for any cloud among {enabled}')
                hint = '\n'.join(f'{c}: {e}' for c, e in errors.items())
                raise ValueError(
                    f'Invalid (region {self._region!r}, zone {self._zone!r}) '
                    f'{where}. Details:\n{hint}')
            if len(valid) > 1:
                raise ValueError(
                    f'Cannot infer cloud from (region {self._region!r}, zone '
                    f'{self._zone!r}). Multiple enabled clouds have '
                    f'region/zone of the same names: {valid}. To fix: '
                    'explicitly specify `cloud`.')
            self._cloud = valid[0]
        self._region, self._zone = self._cloud.validate_region_zone(
            self._region, self._zone)

    def _try_validate_instance_type(self) -> None:
        if self._instance_type is None:
            return
        if self._cloud is not None:
            if not self._cloud.instance_type_exists(self._instance_type):
                raise ValueError(
                    f'Invalid instance type {self._instance_type!r} for '
                    f'cloud {self._cloud}.')
            return
        enabled = sky_check.get_cached_enabled_clouds_or_refresh(
            raise_if_no_cloud_access=True)
        valid = [
            c for c in enabled if c.instance_type_exists(self._instance_type)
        ]
        if not valid:
            where = (f'for cloud {enabled[0]}' if len(enabled) == 1 else
                     f'for any cloud among {enabled}')
            raise ValueError(
                f'Invalid instance type {self._instance_type!r} {where}.')
        if len(valid) > 1:
            raise ValueError(
                f'Ambiguous instance type {self._instance_type!r}. Please '
                f'specify cloud explicitly among {valid}.')
        self._cloud = valid[0]

    def _try_validate_cpus_mem(self) -> None:
        if self._cpus is None and self._memory is None:
            return
        if self._instance_type is None:
            return
        assert self._cloud is not None
        cpus, mem = self._cloud.get_vcpus_mem_from_instance_type(
            self._instance_type)
        for want, have, what in ((self._cpus, cpus, 'vCPUs'),
                                 (self._memory, mem, 'memory')):
            if want is None or have is None:
                continue
            if want.endswith('+'):
                if have < float(want[:-1]):
                    raise ValueError(
                        f'{self._instance_type} does not have enough {what}. '
                        f'{self._instance_type} has {have} {what}, but '
                        f'{want} is requested.')
            elif want.endswith('x'):
                continue
            elif have != float(want):
                raise ValueError(
                    f'{self._instance_type} does not have the requested '
                    f'{what}. {self._instance_type} has {have} {what}, but '
                    f'{want} is requested.')

    def _try_validate_misc(self) -> None:
        if self._max_hourly_cost is not None and self._max_hourly_cost <= 0:
            raise ValueError('max_hourly_cost must be positive. Found: '
                             f'{self._max_hourly_cost}')
        if self._disk_tier is not None and self._cloud is not None and (
                self._disk_tier != resources_utils.DiskTier.BEST):
            ok, msg = self._cloud.check_disk_tier(self._instance_type,
                                                  self._disk_tier)
            if not ok:
                from skypilot_b200 import exceptions  # pylint: disable=import-outside-toplevel
                raise exceptions.NotSupportedError(msg)

    # ---- launchable helpers -----------------------------------------------------
    def is_launchable(self) -> bool:
        return self._cloud is not None and self._instance_type is not None

    def assert_launchable(self) -> 'Resources':
        assert self.is_launchable(), self
        return self

    def is_empty(self) -> bool:
        return all(v is None for v in (
            self._cloud, self._instance_type, self._cpus, self._memory,
            self._accelerators, self._accelerator_args, self._image_id,
            self._disk_tier, self._network_tier, self._ports, self._labels,
            self._local_disk, self._max_hourly_cost)) and (
                not self._use_spot_specified and
                self._disk_size == DEFAULT_DISK_SIZE_GB)

    def get_valid_regions_for_launchable(self) -> List[clouds.Region]:
        """Regions (with zones) that can provision this launchable
        (sky/resources.py:1193-1246)."""
        assert self.is_launchable(), self
        regions = self._cloud.regions_with_offering(self._instance_type,
                                                    self.accelerators,
                                                    self._use_spot,
                                                    self._region, self._zone,
                                                    self)
        allowed = self.allowed_region_names()
        if allowed is not None:
            regions = [r for r in regions if r.name in allowed]
        return regions

    def allowed_region_names(self) -> Optional[Set[str]]:
        """The region allow-list of sky/resources.py:1210-1246, or None: the
        keys of a per-region `image_id` dict, intersected with the keys of a
        per-region `ssh_proxy_command` in the SkyPilot config."""
        from skypilot_b200 import skypilot_config  # pylint: disable=import-outside-toplevel
        allowed: Optional[Set[str]] = None
        if self._image_id is not None and None not in self._image_id:
            allowed = set(self._image_id.keys())
        if self._cloud is not None:
            by_proxy = skypilot_config.allowed_regions_by_ssh_proxy(
                str(self._cloud).lower())
            if by_proxy is not None:
                allowed = by_proxy if allowed is None else allowed & by_proxy
        return allowed

    def get_cost(self, seconds: float) -> float:
        """USD for `seconds` of runtime (sky/resources.py:1685-1698)."""
        hours = seconds / 3600
        assert self._cloud is not None, 'Cloud must be specified'
        assert self._instance_type is not None, (
            'Instance type must be specified')
        hourly_cost = self._cloud.instance_type_to_hourly_cost(
            self._instance_type, self.use_spot, self._region, self._zone)
        if self.accelerators is not None:
            hourly_cost += self._cloud.accelerators_to_hourly_cost(
                self.accelerators, self.use_spot, self._region, self._zone)
        return float(hourly_cost * hours)

    def get_reservations_available_resources(self) -> Dict[str, int]:
        """{reservation name: consumable reserved nodes} of this launchable
        (sky/resources.py:1785-1812); see skypilot_b200/reservations.py."""
        from skypilot_b200 import reservations  # pylint: disable=import-outside-toplevel
        if self.use_spot or isinstance(self._cloud, clouds.DummyCloud):
            return {}
        assert (self._cloud is not None and self._instance_type is not None
                and self._region is not None), (
                    f'Cloud, instance type, region must be specified. '
                    f'Resources={self}')
        return reservations.available_resources(
            str(self._cloud).lower(), self._instance_type, self._region,
            self._zone, self.use_spot)

    def should_be_blocked_by(self, blocked: 'Resources') -> bool:
        """Wildcard match against a blocked entry
        (sky/resources.py:1938-1961): a None field of `blocked` matches
        anything."""
        assert self._cloud is not None, 'Cloud must be specified'
        matched = True
        if (blocked.cloud is not None and
                not self._cloud.is_same_cloud(blocked.cloud)):
            matched = False
        if (blocked.instance_type is not None and
                self.instance_type != blocked.instance_type):
            matched = False
        if blocked.region is not None and self._region != blocked.region:
            matched = False
        if blocked.zone is not None and self._zone != blocked.zone:
            matched = False
        if (blocked.accelerators is not None and
                self.accelerators != blocked.accelerators):
            matched = False
        if blocked.use_spot is not None and self.use_spot != blocked.use_spot:
            matched = False
        return matched

    def extract_docker_image(self) -> Optional[str]:
        if self._image_id is None or len(self._image_id) != 1:
            return None
        image = list(self._image_id.values())[0]
        if image.startswith('docker:'):
            return image[len('docker:'):]
        return None

    def get_required_cloud_features(self) -> Set[Any]:
        """Features a cloud must implement for this request
        (sky/resources.py:2156-2183)."""
        features = set()
        f = clouds.CloudImplementationFeatures
        if self.use_spot:
            features.add(f.SPOT_INSTANCE)
        if (self._disk_tier is not None and
                self._disk_tier != resources_utils.DiskTier.BEST):
            features.add(f.CUSTOM_DISK_TIER)
        if (self._network_tier is not None and
                self._network_tier == resources_utils.NetworkTier.BEST):
            features.add(f.CUSTOM_NETWORK_TIER)
        if self.extract_docker_image() is not None:
            features.add(f.DOCKER_IMAGE)
        elif self._image_id is not None:
            features.add(f.IMAGE_ID)
        if self._ports is not None:
            features.add(f.OPEN_PORTS)
        if self._local_disk is not None:
            features.add(f.LOCAL_DISK)
        return features

    _PLAIN_FIELDS = {
        'cloud': '_cloud', 'instance_type': '_instance_type',
        'region': '_region', 'zone': '_zone', 'labels': '_labels',
        'max_hourly_cost': '_max_hourly_cost', 'job_recovery': '_job_recovery',
    }

    def copy(self, **override) -> 'Resources':
        """A new Resources with some fields replaced
        (sky/resources.py:2076-2143). Fields that need no re-parsing are
        cloned directly; the rest go through the same setters as __init__."""
        new = Resources.__new__(Resources)
        new.__dict__.update(self.__dict__)
        new.__dict__.pop('_validated_store', None)
        new.__dict__.pop('_request_key', None)
        new.__dict__.pop('_plan_templates', None)
        if self._accelerators is not None:
            new._accelerators = dict(self._accelerators)
        for key, value in override.items():
            attr = Resources._PLAIN_FIELDS.get(key)
            if attr is not None:
                setattr(new, attr, value)
            elif key == 'cpus':
                new._set_cpus(value)
            elif key == 'memory':
                new._set_memory(value)
            elif key == 'accelerators':
                new._set_accelerators(value, override.get(
                    'accelerator_args', self._accelerator_args))
            elif key == 'accelerator_args':
                if 'accelerators' not in override:
                    new._accelerator_args = value
            elif key == 'use_spot':
                new._use_spot_specified = value is not None
                new._use_spot = value if value is not None else False
            elif key == 'no_missing_accel_warnings':
                new._no_missing_accel_warnings = value
            elif key in ('disk_size', 'image_id', 'disk_tier', 'network_tier',
                         'local_disk', 'ports', 'infra'):
                # rare: rebuild through the constructor
                return self._copy_via_init(**override)
            else:
                raise AssertionError(f'unknown Resources field {key!r}')
        return new

    def _copy_via_init(self, **override) -> 'Resources':
        use_spot = self._use_spot if self._use_spot_specified else None
        resources = Resources(
            cloud=override.pop('cloud', self._cloud),
            instance_type=override.pop('instance_type', self._instance_type),
            cpus=override.pop('cpus', self._cpus),
            memory=override.pop('memory', self._memory),
            accelerators=override.pop('accelerators', self._accelerators),
            accelerator_args=override.pop('accelerator_args',
                                          self._accelerator_args),
            use_spot=override.pop('use_spot', use_spot),
            job_recovery=override.pop('job_recovery', self._job_recovery),
            disk_size=override.pop('disk_size', self._disk_size),
            region=override.pop('region', self._region),
            zone=override.pop('zone', self._zone),
            image_id=override.pop('image_id', self._image_id),
            disk_tier=override.pop('disk_tier', self._disk_tier),
            network_tier=override.pop('network_tier', self._network_tier),
            local_disk=override.pop('local_disk', self._local_disk),
            max_hourly_cost=override.pop('max_hourly_cost',
                                         self._max_hourly_cost),
            ports=override.pop('ports', self._ports),
            labels=override.pop('labels', self._labels),
            infra=override.pop('infra', None),
            _no_missing_accel_warnings=override.pop(
                'no_missing_accel_warnings', self._no_missing_accel_warnings),
        )
        assert not override, override
        return resources

    # ------------------------------------------------------------------
    # Request alternatives from a YAML-style config (sky/resources.py:
    # 2209-2411): `any_of` / `ordered` lists, several accelerators, and
    # accelerators given by memory size ('32GB+', 'nvidia:16GB:1').
    @classmethod
    def _parse_accelerators_from_str(cls, accelerators: str
                                    ) -> List[Tuple[str, bool]]:
        """-> [(accelerator string, named by the user?)]; a memory-size spec
        expands to every device of that size in common/metadata.csv
        (sky/resources.py:2209-2262)."""
        import re  # pylint: disable=import-outside-toplevel
        from skypilot_b200.utils import accelerator_registry  # pylint: disable=import-outside-toplevel
        assert isinstance(accelerators, str), accelerators
        size = re.compile(r'^[0-9]+[GgMmTt][Bb]\+?$')
        manufacturer = None
        memory = None
        count = 1
        split = accelerators.split(':')
        if len(split) == 3:
            manufacturer, memory, count_str = split
            count = int(count_str)
            assert size.match(memory), \
                'If specifying a GPU manufacturer, you must also' \
                'specify the memory size'
        elif len(split) == 2 and size.match(split[0]):
            memory = split[0]
            count = int(split[1])
        elif len(split) == 2 and size.match(split[1]):
            manufacturer, memory = split
        elif len(split) == 1 and size.match(split[0]):
            memory = split[0]
        else:
            return [(accelerators, True)]
        parsed = resources_utils.parse_memory_resource(memory, 'accelerators',
                                                       allow_plus=True)
        plus = parsed[-1] == '+'
        if plus:
            parsed = parsed[:-1]
        memory_gb = int(parsed)
        return [(f'{device}:{count}', False)
                for device in accelerator_registry.get_devices_by_memory(
                    memory_gb, plus, manufacturer=manufacturer)]

    @classmethod
    def from_yaml_config(cls, config: Optional[Dict[str, Any]]
                        ) -> Union[Set['Resources'], List['Resources']]:
        """A set of Resources for `any_of` (or several accelerators given as
        a set / dict / string), a list for `ordered` (or a list of
        accelerators), else a set with one Resources
        (sky/resources.py:2264-2411)."""
        import collections  # pylint: disable=import-outside-toplevel
        if config is None:
            return {Resources()}
        config = dict(config)

        def aliases(cfg):
            if 'gpus' in cfg:
                if 'accelerators' in cfg:
                    raise ValueError(
                        'Cannot specify both gpus and accelerators in config.')
                cfg['accelerators'] = cfg.pop('gpus')

        aliases(config)
        for key in ('any_of', 'ordered'):
            if isinstance(config.get(key), list):
                config[key] = [dict(c) for c in config[key]]
                for c in config[key]:
                    aliases(c)
                    if 'any_of' in c or 'ordered' in c:
                        raise ValueError(
                            'Invalid resources YAML: "any_of" / "ordered" '
                            'cannot be nested.')

        def override(base, overrides):
            out = []
            for ov in overrides:
                ov = dict(ov)
                new = dict(base)
                ov_labels = ov.pop('labels', None)
                new.update(ov)
                labels = new.get('labels')
                if labels is not None and ov_labels is not None:
                    labels = dict(labels, **ov_labels)
                elif ov_labels is not None:
                    labels = ov_labels
                new['labels'] = labels
                out.extend(list(Resources.from_yaml_config(new)))
            return out

        any_of = config.pop('any_of', None)
        ordered = config.pop('ordered', None)
        if any_of is not None and ordered is not None:
            raise ValueError(
                'Cannot specify both "any_of" and "ordered" in resources.')
        accelerators = config.get('accelerators')
        if config and accelerators is not None:
            if isinstance(accelerators, str):
                parsed = cls._parse_accelerators_from_str(accelerators)
            elif isinstance(accelerators, dict):
                parsed = []
                for k, v in accelerators.items():
                    parsed.extend(cls._parse_accelerators_from_str(
                        f'{k}:{v}' if v is not None else f'{k}'))
            elif isinstance(accelerators, (list, set)):
                parsed = []
                for name in accelerators:
                    parsed.extend(cls._parse_accelerators_from_str(name))
            else:
                raise AssertionError(
                    f'Invalid accelerators type:{type(accelerators)}')
            named: Dict[str, bool] = collections.OrderedDict()
            for accel, user in parsed:
                named[accel] = user or named.get(accel, False)
            kind = list if isinstance(accelerators, list) else set
            accelerators = kind([(a, u) for a, u in named.items()])
            if len(accelerators) > 1 and ordered:
                raise ValueError(
                    'Cannot specify multiple "accelerators" with "ordered" '
                    'in resources.')
            if (len(accelerators) > 1 and any_of and
                    not isinstance(accelerators, set)):
                raise ValueError(
                    'Cannot specify multiple "accelerators" with preferred '
                    'order (i.e., list of accelerators) with "any_of" '
                    'in resources.')
        if any_of:
            return set(override(config, any_of))
        if ordered:
            return override(config, ordered)
        if accelerators:
            out = []
            for acc, user in accelerators:
                one = dict(config)
                one['accelerators'] = acc
                if not user:
                    one['_no_missing_accel_warnings'] = True
                out.append(Resources._from_yaml_config_single(one))
            return type(accelerators)(out)
        return {Resources._from_yaml_config_single(config)}

    _YAML_FIELDS = ('infra', 'region', 'zone', 'instance_type', 'cpus',
                    'memory', 'accelerators', 'accelerator_args', 'use_spot',
                    'job_recovery', 'disk_size', 'image_id', 'disk_tier',
                    'network_tier', 'local_disk', 'max_hourly_cost', 'ports',
                    'labels', '_no_missing_accel_warnings')
    # fields of the reference's schema that do not reach the optimizer path
    _YAML_IGNORED = ('ephemeral_storage', 'autostop', 'priority',
                     'priority_class', 'volumes', '_docker_login_config',
                     '_docker_username_for_runpod', '_is_image_managed',
                     '_requires_fuse', '_cluster_config_overrides')

    @classmethod
    def _from_yaml_config_single(cls, config: Dict[str, Any]) -> 'Resources':
        """sky/resources.py:2413-2489."""
        config = dict(config)
        fields: Dict[str, Any] = {
            'cloud': registry.CLOUD_REGISTRY.from_str(config.pop('cloud',
                                                                 None))
        }
        if config.get('spot_recovery') is not None:
            config['job_recovery'] = config.pop('spot_recovery')
        else:
            config.pop('spot_recovery', None)
        for name in cls._YAML_FIELDS:
            fields[name] = config.pop(name, None)
        for name in cls._YAML_IGNORED:
            config.pop(name, None)
        for name in ('cpus', 'memory', 'disk_size', 'local_disk'):
            if fields[name] is not None:
                fields[name] = str(fields[name])
        if fields['accelerator_args'] is not None:
            fields['accelerator_args'] = dict(fields['accelerator_args'])
        assert not config, f'Invalid resource args: {config.keys()}'
        return Resources(**fields)


class LaunchableResources(Resources):
    """Typing alias: a Resources for which is_launchable() holds."""
