"""Re-point the reference's hot-path symbols at the B200 kernels.

The reference has no plugin/operator API: callers bind the hot-path functions
with ``from X import Y`` at import time (SURVEY.md section 8b).  ``install()``
therefore rebinds the names *in every reference module that imported them*:

  utils.event_process        events_to_voxel_grid(_pol/_pytorch), event_preprocess(_pytorch)
  data_readers.video_readers events_to_voxel_grid, events_to_voxel_grid_pol, event_preprocess
  data_readers.train_data_loaders / data_readers.MVSEC / test_noeval (same names)
  utils.flow_utils           backWarp, forwardWarp, FrameWarp
  e2v.e2v_model, loss        FrameWarp
  loss, test_wo_flow, test_mvsec   voxel_warping_flow_loss (part "fwl")
  data_readers.MVSEC_utils, data_readers.MVSEC, utils.event_uitls (DCEIFlow)
                             eventsToVoxel, eventsToVoxelTorch, events_to_voxel_torch, events_to_neg_pos_voxel_torch
                             (part "mvsec": the second voxeliser)
  ERAFT.corr, ERAFT.eraft    CorrBlock
  DCEIFlow.core.corr.raft_corr, DCEIFlow.DCEIFlow   CorrBlock, AlternateCorrBlock

after which ``model_mode`` 'cista-eiflow' / 'cista-eraft' run unchanged on the
CUDA path.  ``uninstall()`` restores the originals.  The reference checkout must
be importable (on ``sys.path``); modules that are not importable are skipped.
"""
from __future__ import annotations

import importlib
import sys

from . import corr, event_process, flow_utils
from . import loss as loss_mod
from . import mvsec_utils

_VOXEL = {name: getattr(event_process, name) for name in (
    "events_to_voxel_grid", "events_to_voxel_grid_pol", "events_to_voxel_grid_pytorch",
    "event_preprocess", "event_preprocess_pytorch")}
_WARP = {name: getattr(flow_utils, name) for name in ("backWarp", "forwardWarp", "FrameWarp")}
_CORR = {"CorrBlock": corr.CorrBlock, "AlternateCorrBlock": corr.AlternateCorrBlock}
_FWL = {"voxel_warping_flow_loss": loss_mod.voxel_warping_flow_loss}
_MVSEC = {name: getattr(mvsec_utils, name) for name in (
    "eventsToVoxel", "eventsToVoxelTorch", "events_to_voxel_torch", "events_to_neg_pos_voxel_torch")}

# module -> symbols to rebind there (only names the module already has are touched)
TARGETS = {
    "utils.event_process": (_VOXEL,),
    "data_readers.video_readers": (_VOXEL,),
    "data_readers.train_data_loaders": (_VOXEL,),
    "test_noeval": (_VOXEL,),
    "utils.flow_utils": (_WARP,),
    "e2v.e2v_model": (_WARP,),
    "loss": (_WARP, _FWL),
    "test_wo_flow": (_FWL,),
    "test_mvsec": (_FWL,),
    "data_readers.MVSEC_utils": (_MVSEC,),
    "data_readers.MVSEC": (_VOXEL, _MVSEC),
    "DCEIFlow.utils.event_uitls": (_MVSEC,),
    "ERAFT.corr": (_CORR,),
    "ERAFT.eraft": (_CORR,),
    "DCEIFlow.core.corr.raft_corr": (_CORR,),
    "DCEIFlow.DCEIFlow": (_CORR,),
}

_saved: dict[tuple[str, str], object] = {}


def install(import_missing: bool = True, parts=("voxel", "warp", "corr", "fwl", "mvsec")) -> list[str]:
    """Rebind; returns the list of ``module.symbol`` names that were replaced."""
    groups = {"voxel": _VOXEL, "warp": _WARP, "corr": _CORR, "fwl": _FWL, "mvsec": _MVSEC}
    active = [groups[p] for p in parts]
    done = []
    for modname, tables in TARGETS.items():
        tables = [t for t in tables if any(t is a for a in active)]
        if not tables:
            continue
        mod = sys.modules.get(modname)
        if mod is None and import_missing:
            try:
                mod = importlib.import_module(modname)
            except Exception:  # optional deps (h5py, matplotlib ...) or reference not on sys.path
                continue
        if mod is None:
            continue
        for table in tables:
            for name, ours in table.items():
                if hasattr(mod, name) and getattr(mod, name) is not ours:
                    _saved.setdefault((modname, name), getattr(mod, name))
                    setattr(mod, name, ours)
                    done.append(f"{modname}.{name}")
    return done


def uninstall() -> None:
    for (modname, name), orig in list(_saved.items()):
        mod = sys.modules.get(modname)
        if mod is not None:
            setattr(mod, name, orig)
        del _saved[(modname, name)]
