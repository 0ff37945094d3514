from .spaced_sampler import Sampler, SpacedSampler, space_timesteps  # noqa: F401
from .multistep_sampler import DDIMSampler, DPMSolverSampler  # noqa: F401
