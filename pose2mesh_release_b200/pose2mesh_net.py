"""FlatPose2Mesh: drop-in for the reference's ``models.pose2mesh_net`` (lib/models/pose2mesh_net.py:8-29).

    pose3d       = PoseNet(pose2d)                      posenet.LinearModel      (SURVEY.md §8 row f1)
    pose_combine = cat(pose2d, pose3d.detach() / 1000)  fused into the native PoseNet call in eval mode
    cam_mesh     = MeshNet(pose_combine)                meshnet.Pose2Mesh        (rows a1-a9)

``forward`` returns ``(cam_mesh, pose3d)`` like the reference; ``predict_vertices_and_joints`` additionally fuses the
callers' vertex gather and joint regression (lib/core/base.py:130-131; demo/run.py:170-171 — row f2).
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import meshnet, posenet, postprocess


class FlatPose2Mesh(nn.Module):
    def __init__(self, num_joint, graph_L, posenet_pretrained: bool = False):
        super().__init__()
        self.num_joint = num_joint
        # attribute names = the reference's (state_dict prefixes `pose_lifter.` / `pose2mesh.`), constructed in its order
        self.pose_lifter = posenet.LinearModel(num_joint, linear_size=4096, num_stage=2, p_dropout=0.5,
                                               pretrained=posenet_pretrained)
        self.pose2mesh = meshnet.Pose2Mesh(2 + 3, 3, graph_L)

    def _lift(self, pose2d):
        """(pose3d [B, J, 3], pose_combine [B, J, 5]): natively in eval mode, the reference's torch ops otherwise."""
        lifter, flat = self.pose_lifter, pose2d.reshape(len(pose2d), -1)
        if not lifter.training and pose2d.is_cuda and not (torch.is_grad_enabled() and pose2d.requires_grad):
            pose3d, combine = lifter.forward_native(flat, with_combine=True)
            return pose3d.reshape(-1, self.num_joint, 3), combine
        pose3d = lifter(flat).reshape(-1, self.num_joint, 3)
        return pose3d, torch.cat((pose2d, pose3d.detach() / 1000), dim=2)

    def forward(self, pose2d):
        pose3d, combine = self._lift(pose2d)
        return self.pose2mesh(combine), pose3d

    @torch.no_grad()
    def predict_vertices_and_joints(self, pose2d, perm_reverse, n_vertex, joint_regressor):
        """Inference: real vertices [B, n_vertex, 3] (gather fused into MeshNet's head) and regressed joints
        [B, n_joint_out, 3] = joint_regressor @ vertices, plus pose3d."""
        lifter = self.pose_lifter
        pose3d, pose_combine = lifter.forward_native(pose2d.reshape(len(pose2d), -1), with_combine=True)
        verts = self.pose2mesh.forward_vertices(pose_combine, perm_reverse, n_vertex)
        joints = postprocess.regress_joints(verts, joint_regressor)
        return verts, joints, pose3d.reshape(-1, self.num_joint, 3)

    @torch.no_grad()
    def optimize_cam_param(self, joints_px, perm_reverse, n_vertex, joint_regressor, crop_size=500, cam_init=None):
        """demo/run.py:149-197 for B people in one call: joints_px [B, J_in, 2 | 3] image pixels (an integer tensor is
        truncated like the demo's int64 input; a third column is ignored) -> dict of the demo's ``out`` fields,
        batched: ``mesh`` [B, n_vertex, 3], ``cam_param`` [B, 3], ``bbox`` [B, 4] (bbox1), ``target`` [B, J_in, 2],
        plus ``loss`` [B], the L1 loss of each fitted camera.

        Chains normalize_pose2d -> predict_vertices_and_joints -> crop_pose2d -> fit_camera.  Like the demo, the fit
        pairs the regressed joints with the first 17 target joints (run.py:180), so joint_regressor must have 17 rows.
        cam_init=None draws torch.rand((1, 3)) once per person, in order, as the demo's per-person
        project_net.get_model does."""
        from . import project_net

        dev = next(self.parameters()).device
        jp = torch.as_tensor(joints_px)
        if jp.dim() == 2:
            jp = jp[None]
        if jp.dim() != 3 or jp.shape[2] not in (2, 3):
            raise ValueError(f"joints_px must be [B, J, 2 | 3], got {tuple(jp.shape)}")
        n_reg = joint_regressor.shape[0]
        if n_reg != 17 or jp.shape[1] < 17:
            raise ValueError(f"the demo's camera fit pairs 17 regressed joints with the first 17 input joints "
                             f"(demo/run.py:180); got a {n_reg}-row joint_regressor and {jp.shape[1]} input joints")
        B = jp.shape[0]
        if cam_init is None:
            cam_init = torch.cat([torch.rand((1, 3)) for _ in range(B)])
        jp = jp[..., :2].to(dev)
        pose2d = postprocess.normalize_pose2d(jp)
        verts, joints, _ = self.predict_vertices_and_joints(pose2d, perm_reverse, n_vertex, joint_regressor)
        target, bbox = postprocess.crop_pose2d(jp, res=crop_size, aspect_ratio=1.0, scale=1.25)
        cam, loss = project_net.fit_camera(joints, target[:, :17].contiguous(), crop_size, cam_init.to(dev))
        return {"mesh": verts, "cam_param": cam, "bbox": bbox, "target": target, "loss": loss}


def get_model(num_joint, graph_L):
    """lib/models/pose2mesh_net.py:25-28."""
    return FlatPose2Mesh(num_joint, graph_L)
