"""B200-native multi-grid warp (StabNet's transformer / interpolate path) behind the reference's Python interface.

Layout: csrc/ (CUDA kernels + C ABI, built into libmgw_b200.so), _lib.py (ctypes), ops.py (tensor carriers),
functional.py (autograd), spatial_transformer3.py / spatial_transformer.py (reference-named operator modules),
losses.py (vertex builder, loss epilogues, vertex regularisers, schedule, total loss), deploy.py (the deploy loop's pieces: frame
producer, colour-frame warps, history rings, crop), stabnet.py (torch backbone carrier + the reference's objective),
parallel.py (batch sharding + NCCL all-reduce), dropin/ (top-level module names of the reference).
"""
from . import _lib, deploy, functional, losses, ops, parallel, spatial_transformer, spatial_transformer3, stabnet  # noqa: F401
from ._lib import MgwError, launch_count, set_impl  # noqa: F401
from .losses import (feature_loss, get_4_pts, get_black_pos, get_black_pos_loss, get_consistency_loss, get_distortion_loss,  # noqa: F401
                     img_loss, loss_gates, pass_coef, temp_loss, total_loss, train_pass, transformer_img_loss, vertex_losses)
from .deploy import CropState, MixedStreamBatch, PlaneTable, StreamBatch, StreamState, warpRevBundle, warpRevBundle2  # noqa: F401
from .spatial_transformer import interpolate  # noqa: F401
from .stabnet import StabNet, inference_stable_net, train_losses  # noqa: F401
from .spatial_transformer3 import transformer  # noqa: F401

__version__ = '0.1.0'
