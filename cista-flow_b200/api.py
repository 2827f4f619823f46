"""Public surface of the package (re-exported by ``cistaflow_b200``)."""
from ._lib import CistaFlowError, LIB_PATH, load as load_library
from .corr import AlternateCorrBlock, CorrBlock, build_pyramid, coords_grid, lookup as corr_lookup
from .event_process import (event_preprocess, event_preprocess_batched, event_preprocess_pytorch,
                            events_to_voxel_grid, events_to_voxel_grid_batched, events_to_voxel_grid_packed,
                            events_to_voxel_grid_pol, events_to_voxel_grid_pytorch, filter_events, pack_events,
                            pack_events_host, window_offsets)
from .flow_utils import (FrameWarp, backWarp, flow_any, forwardWarp, warp, warp_frame_and_codes,
                         warp_frame_and_codes_upflow8)
from .install import install, uninstall
from .loss import voxel_warping_flow_loss
from .mvsec_utils import eventsToVoxel, eventsToVoxelTorch, events_to_neg_pos_voxel_torch, events_to_voxel_torch

__all__ = [
    "CistaFlowError", "LIB_PATH", "load_library",
    "AlternateCorrBlock", "CorrBlock", "build_pyramid", "coords_grid", "corr_lookup",
    "event_preprocess", "event_preprocess_batched", "event_preprocess_pytorch",
    "events_to_voxel_grid", "events_to_voxel_grid_batched", "events_to_voxel_grid_packed", "events_to_voxel_grid_pol",
    "events_to_voxel_grid_pytorch", "pack_events", "pack_events_host", "filter_events", "window_offsets",
    "FrameWarp", "backWarp", "flow_any", "forwardWarp", "warp", "warp_frame_and_codes", "warp_frame_and_codes_upflow8",
    "install", "uninstall", "voxel_warping_flow_loss",
    "eventsToVoxel", "eventsToVoxelTorch", "events_to_neg_pos_voxel_torch", "events_to_voxel_torch",
]
