"""skypilot_b200: SkyPilot's placement optimizer hot path on B200 GPUs.

Drop-in surface (same names as the `sky` package for this path):
`Resources`, `Task`, `Dag`, `Optimizer`, `OptimizeTarget`, `clouds`,
`catalog`, `optimize`. Everything row-level runs in hand-written sm_100a CUDA
kernels behind `libskyopt.so` (include/skyopt.h); see DESIGN.md.
"""
from skypilot_b200 import catalog
from skypilot_b200 import check
from skypilot_b200 import clouds
from skypilot_b200 import exceptions
from skypilot_b200 import reservations
from skypilot_b200.dag import Dag
from skypilot_b200.optimizer import DummyResources
from skypilot_b200.optimizer import Optimizer
from skypilot_b200.optimizer import OptimizeTarget
from skypilot_b200.resources import Resources
from skypilot_b200.task import Task

AWS = clouds.AWS
GCP = clouds.GCP
Azure = clouds.Azure
Lambda = clouds.Lambda

optimize = Optimizer.optimize
optimize_batch = Optimizer.optimize_batch

__version__ = '0.1.0'

__all__ = [
    'AWS', 'Azure', 'Dag', 'DummyResources', 'GCP', 'Lambda', 'Optimizer',
    'OptimizeTarget', 'Resources', 'Task', 'catalog', 'check', 'clouds',
    'exceptions', 'optimize', 'optimize_batch', 'reservations'
]
