"""The steps either side of the model in the reference's callers, on the GPU (SURVEY.md §8 row f2):

    regress_joints(verts, J)      lib/core/base.py:131,204; demo/run.py:171   joints = J_regressor @ vertices
    normalize_pose2d(joints_px)   demo/run.py:150-158                          pixels -> network input coordinates
    crop_pose2d(joints_px)        demo/run.py:150-153                          pixels -> camera-fit target + bbox1

All run in libp2m_b200.so (p2m_regress_joints, p2m_normalize_pose2d, p2m_crop_pose2d); CUDA tensors only.
"""
from __future__ import annotations

import torch

from . import _lib

INPUT_SHAPE = (384, 288)  # cfg.MODEL.input_shape (height, width), lib/core/config.py:52


def regress_joints(vertices: torch.Tensor, joint_regressor: torch.Tensor) -> torch.Tensor:
    """vertices [B, n_vertex, C] (C <= 4), joint_regressor [n_joint, n_vertex] -> joints [B, n_joint, C]."""
    if not vertices.is_cuda:
        raise RuntimeError("pose2mesh_release_b200 runs on CUDA (sm_100a) only; got a CPU tensor")
    v = vertices.contiguous().float()
    jr = joint_regressor.to(v.device).contiguous().float()
    B, nv, ch = v.shape
    if jr.shape[1] != nv:
        raise ValueError(f"joint_regressor has {jr.shape[1]} columns, vertices has {nv} rows")
    out = torch.empty((B, jr.shape[0], ch), device=v.device, dtype=torch.float32)
    with torch.cuda.device(v.device):
        _lib.check(_lib.load().p2m_regress_joints(jr.data_ptr(), v.data_ptr(), out.data_ptr(), B, jr.shape[0], nv, ch,
                                                  torch.cuda.current_stream(v.device).cuda_stream), "p2m_regress_joints")
    return out


def normalize_pose2d(joints_px: torch.Tensor, input_shape=INPUT_SHAPE) -> torch.Tensor:
    """joints_px [B, J, 2] (or [J, 2]) image pixels on a CUDA device -> pose2d [B, J, 2] as demo/run.py:150-158
    computes it.  Integer tensors are treated like the reference treats integer arrays (its in-place affine transform
    truncates the transformed coordinates, aug_utils.py:57-59)."""
    if not joints_px.is_cuda:
        raise RuntimeError("pose2mesh_release_b200 runs on CUDA (sm_100a) only; got a CPU tensor")
    truncate = int(not joints_px.is_floating_point())
    x = joints_px.reshape(-1, joints_px.shape[-2], 2).contiguous().float()
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(_lib.load().p2m_normalize_pose2d(x.data_ptr(), out.data_ptr(), x.shape[0], x.shape[1],
                                                    int(input_shape[0]), int(input_shape[1]), truncate,
                                                    torch.cuda.current_stream(x.device).cuda_stream),
                   "p2m_normalize_pose2d")
    return out


def crop_pose2d(joints_px: torch.Tensor, res: int = 500, aspect_ratio: float = 1.0, scale: float = 1.25):
    """joints_px [B, J, 2] (or [J, 2]; J <= 32) image pixels on a CUDA device -> (joints [B, J, 2] in pixels of the
    res x res patch, bbox [B, 4] = [x, y, w, h]): the camera fit's target and the box the demo calls bbox1
    (demo/run.py:150-153: get_bbox, process_bbox(aspect_ratio=1.0, scale=1.25), j2d_processing).  Integer tensors
    are truncated like in normalize_pose2d."""
    if not joints_px.is_cuda:
        raise RuntimeError("pose2mesh_release_b200 runs on CUDA (sm_100a) only; got a CPU tensor")
    truncate = int(not joints_px.is_floating_point())
    x = joints_px.reshape(-1, joints_px.shape[-2], 2).contiguous().float()
    out = torch.empty_like(x)
    bbox = torch.empty((x.shape[0], 4), device=x.device, dtype=torch.float32)
    with torch.cuda.device(x.device):
        _lib.check(_lib.load().p2m_crop_pose2d(x.data_ptr(), out.data_ptr(), bbox.data_ptr(), x.shape[0], x.shape[1],
                                               int(res), int(res), float(aspect_ratio), float(scale), truncate,
                                               torch.cuda.current_stream(x.device).cuda_stream), "p2m_crop_pose2d")
    return out, bbox
