"""vbnn_b200 -- the VBLinear hot path of louissmit/VBNN on B200 (sm_100a).

Host-side mirror of the reference's Torch7 interface over libvbnn.so (include/vbnn.h).  Importing
the package never touches the GPU; the first object constructed loads libvbnn.so and fails loudly
if it is missing (there is no CPU / PyTorch fallback)."""
from . import _lib
from ._lib import VbnnError, knob, lib
from .config import default_opt, opts_struct
from .context import Context, default_context
from .mlp import MLP, OutputPrediction, Prediction
from .vblinear import Linear, VBLinear

__all__ = ["VbnnError", "lib", "knob", "default_opt", "opts_struct", "Context", "default_context", "MLP",
           "OutputPrediction", "Prediction", "VBLinear", "Linear"]
