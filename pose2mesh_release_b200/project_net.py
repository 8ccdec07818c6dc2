"""The demo's weak-perspective camera: drop-in for the reference's ``models.project_net`` (lib/models/project_net.py)
plus the camera fit of demo/run.py:160-189 on the GPU (SURVEY.md §8 row f5).

    OptimzeCamLayer(crop_size)     project_net.py:6-17   out = (p[:, :, :2] + c[1:]) * c[0] * R + R,  R = crop_size / 2
    OptimzeCamLayer.fit(...)       run.py:172-186        the layer's camera fitted natively (p2m_fit_camera)
    fit_camera(...)                run.py:172-186        the same fit for B people in one launch, one warp per person
    convert_crop_cam_to_orig_img   run.py:24-43          crop camera -> camera of the original image

The reference fits one person with 1500 Python-level steps of nn.L1Loss + optim.Adam (lr 0.1, 0.05 after loop index
500, 0.001 after 1000): a few dozen tiny launches per step.  ``p2m_fit_camera`` keeps a person's camera and Adam state
in the registers of one warp for all the steps, so a whole crowd is one launch.  CUDA tensors only.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import _lib


class OptimzeCamLayer(nn.Module):
    """lib/models/project_net.py:6-17 (name, ``img_res``, the single ``cam_param`` Parameter and its
    ``torch.rand((1, 3))`` draw at construction are the reference's, so RNG consumption is identical)."""

    def __init__(self, crop_size):
        super().__init__()
        self.img_res = crop_size / 2
        self.cam_param = nn.Parameter(torch.rand((1, 3)))

    def forward(self, pose3d):
        output = pose3d[:, :, :2] + self.cam_param[None, :, 1:]
        output = output * self.cam_param[None, :, :1] * self.img_res + self.img_res
        return output

    @torch.no_grad()
    def fit(self, pose3d: torch.Tensor, target: torch.Tensor, iters: int = 1500) -> torch.Tensor:
        """Fit ``cam_param`` to the 2-D target as demo/run.py:172-186 does, natively: pose3d [1, J, >=2] (or [J, >=2]),
        target [1, J, 2] (or [J, 2]) on a CUDA device.  Starts from the current ``cam_param``, writes the fitted
        camera back into it and returns the L1 loss of the fitted camera (a 0-dim tensor)."""
        if not (pose3d.is_cuda and target.is_cuda):
            raise RuntimeError("OptimzeCamLayer.fit runs on CUDA (sm_100a) only; got a CPU tensor")
        p = pose3d.reshape(1, pose3d.shape[-2], pose3d.shape[-1])
        t = target.reshape(1, target.shape[-2], target.shape[-1])
        cam, loss = fit_camera(p, t, 2 * self.img_res, self.cam_param.detach().to(p.device).reshape(1, 3), iters)
        self.cam_param.copy_(cam.to(self.cam_param.device))
        return loss[0]


def get_model(crop_size):
    """lib/models/project_net.py:20-23."""
    return OptimzeCamLayer(crop_size)


def fit_camera(joints3d: torch.Tensor, target: torch.Tensor, crop_size, cam_init: torch.Tensor, iters: int = 1500):
    """joints3d [B, J, >=2] (x, y used), target [B, J, 2] in crop pixels, cam_init [B, 3] -> (cam [B, 3], loss [B]):
    per person, ``iters`` steps of the demo's fit (mean L1 loss + Adam with its lr schedule) from cam_init, and the L1
    loss of the fitted camera.  J <= 32.  All on one CUDA device."""
    if not (joints3d.is_cuda and target.is_cuda and cam_init.is_cuda):
        raise RuntimeError("fit_camera runs on CUDA (sm_100a) only; got a CPU tensor")
    if joints3d.dim() != 3 or joints3d.shape[2] < 2:
        raise ValueError(f"joints3d must be [B, J, >=2], got {tuple(joints3d.shape)}")
    B, J = joints3d.shape[:2]
    if tuple(target.shape) != (B, J, 2):
        raise ValueError(f"target must be [{B}, {J}, 2] to pair with joints3d, got {tuple(target.shape)}")
    if tuple(cam_init.shape) != (B, 3):
        raise ValueError(f"cam_init must be [{B}, 3], got {tuple(cam_init.shape)}")
    dev = joints3d.device
    p = joints3d.contiguous().float()
    t = target.to(dev).contiguous().float()
    c = cam_init.to(dev).contiguous().float()
    cam = torch.empty((B, 3), device=dev, dtype=torch.float32)
    loss = torch.empty((B,), device=dev, dtype=torch.float32)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().p2m_fit_camera(p.data_ptr(), t.data_ptr(), c.data_ptr(), cam.data_ptr(), loss.data_ptr(),
                                              B, J, p.shape[2], float(crop_size), int(iters),
                                              torch.cuda.current_stream(dev).cuda_stream), "p2m_fit_camera")
    return cam, loss


def convert_crop_cam_to_orig_img(cam: torch.Tensor, bbox: torch.Tensor, img_width, img_height) -> torch.Tensor:
    """demo/run.py:24-43: camera [B, 3] of the crop around bbox [B, 4] = [x, y, w, h] -> [B, 4] = (sx, sy, tx, ty)
    of the original img_width x img_height image."""
    x, y, w, h = bbox[:, 0], bbox[:, 1], bbox[:, 2], bbox[:, 3]
    cx, cy = x + w / 2, y + h / 2
    hw, hh = img_width / 2., img_height / 2.
    sx = cam[:, 0] * (1. / (img_width / h))
    sy = cam[:, 0] * (1. / (img_height / h))
    tx = ((cx - hw) / hw / sx) + cam[:, 1]
    ty = ((cy - hh) / hh / sy) + cam[:, 2]
    return torch.stack([sx, sy, tx, ty], dim=1)
