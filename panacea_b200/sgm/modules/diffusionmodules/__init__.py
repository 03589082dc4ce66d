from .controlmodel import ControlledUNetModel3D, ControlNet3D  # noqa: F401
from .denoiser import DiscreteDenoiser  # noqa: F401
from .discretizer import EDMDiscretization, LegacyDDPMDiscretization  # noqa: F401
from .guiders import VanillaCFG  # noqa: F401
from .sampling import (DPMPP2MSampler, DPMPP2SAncestralSampler, EulerAncestralSampler, EulerEDMSampler,  # noqa: F401
                       HeunEDMSampler, LinearMultistepSampler)
from .wrappers import OpenAIWrapperControlLDM3D  # noqa: F401
