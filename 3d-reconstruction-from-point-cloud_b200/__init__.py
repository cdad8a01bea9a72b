"""points_transfer_b200 -- B200-native (sm_100a) drop-in for the pointsTransfer
detail-transfer hot path of horizon-research/3D-Reconstruction-From-Point-Cloud.

Import with ``importlib.import_module("3d-reconstruction-from-point-cloud_b200")`` (the
directory name is not a Python identifier) or through ``__graft_entry__.package()``.
"""
from .api import (  # noqa: F401
    ABI_SYMBOLS, SYNTH_SYMBOLS, ATTR_DTYPE, CAND_DTYPE, COORD_AUTO, COORD_F32, COORD_F64, LIB_PATH,
    POINT_DTYPE, PT_MAX_K, DeviceTree, Distance, K_neighbor_search, PointsTransferError, ShardedTree, Tree, texture_from_lists,
    bake_compose_device, bake_compose_height_device, bake_compose_tangent_device, bake_frames_device,
    bake_samples_device, bake_texels_device,
    device_count, get_option, kernel_launch_count, lib, synth_lib,
    make_points, merge_device, set_option,
    status_string, version,
)
from . import synth  # noqa: F401
from . import dist  # noqa: F401,E402
from . import sharded  # noqa: F401,E402
