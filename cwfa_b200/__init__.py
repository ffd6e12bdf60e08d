"""cwfa_b200 -- B200-native (sm_100a) implementation of the CWFA conditional-wavelet-flow hot path.

Drop-in surface (same names / signatures / state_dict keys as the reference, pvjosue/CWFA):
    cwfa_b200.framework  ~ FrEIA.framework   (Node, InputNode, ConditionNode, OutputNode, GraphINN, SequenceINN)
    cwfa_b200.modules    ~ FrEIA.modules + INN_utils (HaarTransform1D, PermuteDim, HaarDownsampling, Split, ...)
    cwfa_b200.networks   ~ networks.py + unet.py (conditional_wavelet_flow, cond_network, Encoder, ...)
    cwfa_b200.pipeline   ~ the ~40 lines of CWFA.py that drive the flow (reconstruct / forward NLL)
All arithmetic runs in hand-written CUDA kernels behind the C ABI in include/cwfa_b200.h.
"""
from . import _lib, data, framework, modules, networks, ops, packed  # noqa: F401
from .data import LensletLayout  # noqa: F401
from .packed import inference_precision, set_inference_precision, weights_changed  # noqa: F401
from .pipeline import CWFAModel, CWFAConfig  # noqa: F401

__version__ = "0.1.0"


def lib_path() -> str:
    return _lib.lib_path()
