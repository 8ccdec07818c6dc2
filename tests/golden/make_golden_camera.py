#!/usr/bin/env python
"""Golden vectors for the demo's camera fit, produced by the UNMODIFIED reference modules in the build container:

    python tests/golden/make_golden_camera.py      ->  tests/golden/camera_fit.npz

  crop_input / crop_target / crop_bbox   run.py:150-153 with the reference's get_bbox, process_bbox(aspect_ratio=1.0,
                                         scale=1.25) and j2d_processing into the 500 x 500 patch: case 0 is
                                         demo/h36m_joint_input.npy (int64: truncated), cases 1.. seeded float poses
                                         (float32 values, passed to the reference as float64 like the demo's arrays)
  init_seeds / init_cam                  project_net.get_model(500).cam_param after torch.manual_seed(s)
  fwd_in / fwd_out                       project_net.OptimzeCamLayer.forward on a fixed input
  fit_joints3d / fit_cam_init            3-D joints (oracle.camera_oracle.synthetic_case) and the starting camera
                                         (torch.manual_seed(1000 + case); get_model(500)) of each fit case
  fit_cam_<k>, fit_loss                  the camera after k = 1, 10, 50, 1500 steps of run.py:172-186 (nn.L1Loss +
                                         optim.Adam, the reference's lr schedule) and the L1 loss of the final camera
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import camera_oracle as co  # noqa: E402
from oracle import ref_shim  # noqa: E402

N_FLOAT = 31
STEPS = (1, 10, 50, 1500)


def main():
    ref_shim.load("human36")
    import aug_utils  # noqa: E402  (reference modules)
    import coord_utils  # noqa: E402
    from models import project_net  # noqa: E402

    demo = np.load(os.path.join(ref_shim.REF_ROOT, "demo", "h36m_joint_input.npy"))
    poses = co.seeded_poses(N_FLOAT, seed=21)
    inputs = [demo] + [p.astype(np.float64) for p in poses]
    targets, bboxes = [], []
    for joint_input in inputs:                                               # run.py:150-153
        bbox = coord_utils.get_bbox(joint_input)
        bbox1 = coord_utils.process_bbox(bbox.copy(), aspect_ratio=1.0, scale=1.25)
        tgt, _ = aug_utils.j2d_processing(joint_input.copy(), (500, 500), bbox1, 0, 0, None)
        targets.append(tgt[:, :2].astype(np.float32))
        bboxes.append(np.asarray(bbox1, dtype=np.float32))
    targets, bboxes = np.stack(targets), np.stack(bboxes)

    seeds = np.arange(8)
    init = []
    for s in seeds:
        torch.manual_seed(int(s))
        init.append(project_net.get_model(500).cam_param.detach()[0].numpy().copy())
    torch.manual_seed(7)
    layer = project_net.get_model(500)
    fwd_in = torch.randn(2, 17, 3, generator=torch.Generator().manual_seed(8))
    with torch.no_grad():
        fwd_out = layer(fwd_in)

    j3d, cam0, snaps, losses = [], [], {k: [] for k in STEPS}, []
    for c, tgt in enumerate(targets):
        p3 = torch.from_numpy(co.synthetic_case(tgt, seed=500 + c))[None]
        torch.manual_seed(1000 + c)
        net = project_net.get_model(500)
        j3d.append(p3[0].numpy())
        cam0.append(net.cam_param.detach()[0].numpy().copy())
        target = torch.from_numpy(tgt)[None]
        criterion = torch.nn.L1Loss()                                        # run.py:163-164
        optimizer = torch.optim.Adam(net.parameters(), lr=0.1)
        net.train()
        for j in range(0, 1500):                                             # run.py:172-186
            pred = net(p3.detach())
            loss = criterion(pred, target[:, :17, :])
            optimizer.zero_grad()
            loss.backward()
            optimizer.step()
            if j == 500:
                for param_group in optimizer.param_groups:
                    param_group["lr"] = 0.05
            if j == 1000:
                for param_group in optimizer.param_groups:
                    param_group["lr"] = 0.001
            if j + 1 in snaps:
                snaps[j + 1].append(net.cam_param.detach()[0].numpy().copy())
        with torch.no_grad():
            losses.append(float(criterion(net(p3), target)))
    out = os.path.join(HERE, "camera_fit.npz")
    np.savez_compressed(out, crop_input=np.stack([i.astype(np.float64) for i in inputs]), crop_input_is_int=np.array(
        [1] + [0] * N_FLOAT), crop_target=targets, crop_bbox=bboxes, init_seeds=seeds, init_cam=np.stack(init),
        fwd_seed=np.array(7), fwd_in=fwd_in.numpy(), fwd_out=fwd_out.numpy(), fit_joints3d=np.stack(j3d),
        fit_cam_init=np.stack(cam0), fit_loss=np.array(losses, dtype=np.float32),
        **{f"fit_cam_{k}": np.stack(v) for k, v in snaps.items()})
    print("wrote", out, os.path.getsize(out), "bytes")


if __name__ == "__main__":
    main()
