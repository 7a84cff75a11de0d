from .base_ray_trafo import BaseRayTrafo
from .geometry import ParallelBeamGeometry2D
from .b200_ray_trafo import B200RayTrafo, NormalOp, MeasurementWeights
from .simulation import simulate, simulate_poisson, SimulatedDataset

# the reference's name for the 2-D parallel-beam operator (src/physics/trafo.py:16)
SimpleTrafo = B200RayTrafo
