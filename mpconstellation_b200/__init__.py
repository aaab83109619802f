"""mpconstellation_b200 -- B200 (sm_100a) implementation of mpconstellation's batched SCvx
linearize-and-discretize step and nonlinear orbit propagation, behind the reference's own
Discretizer / Simulator call signatures.  FP64 CUDA kernels through a C-ABI; no CPU fallback."""
from . import _lib
from ._lib import pinned_empty
from ._numa import bind_host_to_gpu
from .atmosphere import Atmosphere, fit_atmosphere
from .conjunctions import Conjunctions, screen_conjunctions, screen_conjunctions_device
from .batch import (DiscretizedBatch, discretize_batch, discretize_batch_device, fp64_peak_tflops, launch_count,
                    propagate_batch, propagate_batch_device, propagate_discretize, propagate_discretize_device)
from .constraints import (DynamicsJacobian, constraint_terms_batch, constraint_terms_device, dynamics_jacobian,
                          dynamics_jacobian_device, get_constraint_terms)
from .control import (ConstantTangentialThrustController, ConstantThrustController, Controller, ControllerSpec,
                      SequenceController, spec_from)
from .discretizer import Discretizer
from .model import Constants, Satellite, SatelliteScale
from .simulator import Simulator

__all__ = ["Atmosphere", "fit_atmosphere", "Discretizer", "Simulator", "Satellite", "SatelliteScale", "Constants", "Controller",
           "ConstantThrustController", "ConstantTangentialThrustController", "SequenceController", "ControllerSpec",
           "spec_from", "discretize_batch", "discretize_batch_device", "propagate_batch", "propagate_batch_device",
           "propagate_discretize", "propagate_discretize_device", "constraint_terms_batch", "constraint_terms_device", "get_constraint_terms", "dynamics_jacobian", "dynamics_jacobian_device", "DynamicsJacobian", "DiscretizedBatch", "pinned_empty", "bind_host_to_gpu", "fp64_peak_tflops", "launch_count",
           "Conjunctions", "screen_conjunctions", "screen_conjunctions_device"]
