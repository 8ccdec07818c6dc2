"""TEST INFRASTRUCTURE ONLY — CPU restatement of the demo's camera fit.

Only tests/, tools/ and __graft_entry__ may import this package.

    lib/models/project_net.py:6-23        OptimzeCamLayer: out = (p[:, :, :2] + c[1:]) * c[0] * R + R, R = crop_size / 2
    demo/run.py:150-153                   projection target: get_bbox -> process_bbox(aspect_ratio=1.0, scale=1.25) ->
                                          j2d_processing into the crop_size x crop_size patch (bbox1)
    demo/run.py:163-164,172-186           nn.L1Loss + optim.Adam(lr=0.1), 1500 steps, lr 0.05 after loop index 500 and
                                          0.001 after 1000; one person at a time, fp32

The loop is the reference's, op for op, on whatever device its tensors are on (tools/bench_camera_fit.py times it on
CUDA tensors as the demo runs it).  Parity status: PINNED — tests/golden/camera_fit.npz holds what the unmodified
reference's modules compute (tests/golden/make_golden_camera.py); tests/test_camera_cpu.py checks this file against it.
"""
from __future__ import annotations

from typing import Dict, Sequence, Tuple

import numpy as np
import torch
import torch.nn as nn
import torch.optim as optim

from . import demo_oracle as do

CROP_SIZE = 500  # virtual_crop_size, demo/run.py:197


class CamLayer(nn.Module):
    """project_net.py:6-17."""

    def __init__(self, crop_size):
        super().__init__()
        self.img_res = crop_size / 2
        self.cam_param = nn.Parameter(torch.rand((1, 3)))

    def forward(self, pose3d):
        output = pose3d[:, :, :2] + self.cam_param[None, :, 1:]
        output = output * self.cam_param[None, :, :1] * self.img_res + self.img_res
        return output


def crop_target(joint_input: np.ndarray, crop_size: int = CROP_SIZE) -> Tuple[np.ndarray, np.ndarray]:
    """run.py:150-153: (target [J, 2] float32 in patch pixels, bbox1 [4] float32).  Integer input is truncated like
    the reference's in-place transform of the demo's int64 array (demo_oracle.j2d_processing)."""
    bbox1 = do.process_bbox(do.get_bbox(joint_input).copy(), aspect_ratio=1.0, scale=1.25)
    target = do.j2d_processing(joint_input.copy(), (crop_size, crop_size), bbox1)[:, :2]
    return target.astype(np.float32), np.asarray(bbox1, dtype=np.float32)


def fit_camera(pose3d: torch.Tensor, target: torch.Tensor, cam_init: torch.Tensor, crop_size=CROP_SIZE,
               iters: int = 1500, record: Sequence[int] = ()) -> Tuple[torch.Tensor, float, Dict[int, torch.Tensor]]:
    """run.py:172-186 for one person: pose3d [J, >=2], target [J, 2], cam_init [3] (or [1, 3]) -> (camera [3], L1 loss
    of that camera, {step: camera after that many steps for step in record})."""
    net = CamLayer(crop_size).to(pose3d.device)
    with torch.no_grad():
        net.cam_param.copy_(cam_init.reshape(1, 3))
    p, t = pose3d[None].float(), target[None].float()
    criterion = nn.L1Loss()
    optimizer = optim.Adam(net.parameters(), lr=0.1)
    snaps = {}
    net.train()
    for j in range(iters):
        pred = net(p.detach())
        loss = criterion(pred, t)
        optimizer.zero_grad()
        loss.backward()
        optimizer.step()
        if j == 500:
            for g in optimizer.param_groups:
                g["lr"] = 0.05
        if j == 1000:
            for g in optimizer.param_groups:
                g["lr"] = 0.001
        if j + 1 in record:
            snaps[j + 1] = net.cam_param.detach()[0].clone()
    with torch.no_grad():
        final = float(criterion(net(p), t))
    return net.cam_param.detach()[0].clone(), final, snaps


def fit_cameras(joints3d: torch.Tensor, target: torch.Tensor, cam_init: torch.Tensor, crop_size=CROP_SIZE,
                iters: int = 1500) -> Tuple[torch.Tensor, torch.Tensor]:
    """fit_camera person by person: joints3d [B, J, >=2], target [B, J, 2], cam_init [B, 3] -> (cam [B, 3], loss [B])."""
    cams, losses = [], []
    for b in range(joints3d.shape[0]):
        c, l, _ = fit_camera(joints3d[b], target[b], cam_init[b], crop_size, iters)
        cams.append(c)
        losses.append(l)
    return torch.stack(cams), torch.tensor(losses)


def fit_cameras_batched(joints3d: torch.Tensor, target: torch.Tensor, cam_init: torch.Tensor, crop_size=CROP_SIZE,
                        iters: int = 1500) -> Tuple[torch.Tensor, torch.Tensor]:
    """fit_cameras with the people stacked into one [B, 1, 3] parameter: the sum of the per-person mean-L1 losses
    gives every person the gradient of its own loss, and Adam is elementwise, so each person follows the loop above
    (tests/test_camera_cpu.py checks the two agree); one pass of torch ops per step instead of B."""
    r = crop_size / 2
    cam = nn.Parameter(cam_init.reshape(-1, 1, 3).float().clone())
    p, t = joints3d.float().detach(), target.float()
    optimizer = optim.Adam([cam], lr=0.1)

    def per_person_loss():
        out = (p[:, :, :2] + cam[:, :, 1:]) * cam[:, :, :1] * r + r
        return (out - t).abs().mean(dim=(1, 2))

    for j in range(iters):
        loss = per_person_loss().sum()
        optimizer.zero_grad()
        loss.backward()
        optimizer.step()
        if j == 500:
            for g in optimizer.param_groups:
                g["lr"] = 0.05
        if j == 1000:
            for g in optimizer.param_groups:
                g["lr"] = 0.001
    with torch.no_grad():
        return cam.detach()[:, 0].clone(), per_person_loss()


def project(pose3d: torch.Tensor, cam: torch.Tensor, crop_size=CROP_SIZE) -> torch.Tensor:
    """The layer's forward for a batch of cameras: pose3d [B, J, >=2], cam [B, 3] -> [B, J, 2] (fp64 for comparing)."""
    p, c, r = pose3d[..., :2].double(), cam.double(), crop_size / 2
    return (p + c[:, None, 1:]) * c[:, None, :1] * r + r


def synthetic_case(target: np.ndarray, seed: int, crop_size=CROP_SIZE) -> np.ndarray:
    """Plausible 3-D joints [J, 3] for a target: a known camera (scale 0.6-1.2, translation +-0.2) inverted on the
    target, plus seeded noise in xy (sd 0.03) and z (sd 0.15)."""
    g = np.random.default_rng(seed)
    r = crop_size / 2
    s, t = g.uniform(0.6, 1.2), g.uniform(-0.2, 0.2, 2)
    xy = (target.astype(np.float64) - r) / (s * r) - t + g.normal(0, 0.03, target.shape)
    z = g.normal(0, 0.15, (target.shape[0], 1))
    return np.concatenate([xy, z], axis=1).astype(np.float32)


def seeded_poses(n: int, seed: int, n_joint: int = 17) -> np.ndarray:
    """n float32 2-D poses in pixels (the layout tests/test_gpu_front_back.py uses for normalize_pose2d)."""
    g = np.random.default_rng(seed)
    return (g.uniform(0, 1, (n, n_joint, 2)) * np.array([640.0, 480.0]) + g.uniform(0, 300, (n, 1, 2))).astype(np.float32)
