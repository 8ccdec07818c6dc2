#!/usr/bin/env python
"""Timing of the demo's camera fit (GPU box): prints one JSON line.

    python tools/bench_camera_fit.py [--out profiles/camera_fit_b200.json]

  fit_camera_ms[B]        device time (CUDA events) of one p2m_fit_camera launch, 1500 steps, B = 1, 8, 256, 4096;
                          median of 20 runs after 3 warm-up runs
  reference_loop_ms       the reference's per-person loop (nn.L1Loss + optim.Adam, 1500 steps, restated in
                          oracle/camera_oracle.py) on CUDA tensors at B = 1 as the demo runs it; wall time, median of 3
  demo_8_people_ms        8 people end to end on the SMPL-size fixture graph (6890 vertices): one
                          FlatPose2Mesh.optimize_cam_param call against 8 demo-style calls (B = 1 network, then the
                          reference's loop); wall time, median of 3
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402


def power_limit_w():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return float(q.stdout.strip().splitlines()[0]) if q.returncode == 0 else "not measured"
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        return "not measured"


def device_ms(fn, n=20, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def wall_ms(fn, n=3):
    fn()
    ts = []
    for _ in range(n):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()

    from helpers import graph_from_fixture
    from oracle import camera_oracle as co
    from pose2mesh_release_b200 import pose2mesh_net, postprocess, project_net

    dev = torch.device("cuda:0")
    res = {"device": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(), "iters": 1500}

    poses = co.seeded_poses(4096, seed=1)
    tgt = torch.from_numpy(np.stack([co.crop_target(p.astype(np.float64))[0] for p in poses[:256]]))
    tgt = tgt.repeat(16, 1, 1)
    j3 = torch.from_numpy(np.stack([co.synthetic_case(t.numpy(), i) for i, t in enumerate(tgt[:256])])).repeat(16, 1, 1)
    c0 = torch.rand(4096, 3, generator=torch.Generator().manual_seed(2))
    j3, tgt, c0 = j3.to(dev), tgt.to(dev), c0.to(dev)
    res["fit_camera_ms"] = {str(b): device_ms(lambda b=b: project_net.fit_camera(j3[:b], tgt[:b], 500, c0[:b]))
                            for b in (1, 8, 256, 4096)}
    res["reference_loop_ms_per_person"] = wall_ms(lambda: co.fit_camera(j3[0], tgt[0], c0[0]))

    mats, zg = graph_from_fixture("smpl_like")
    perm_rev = np.asarray(zg["perm_reverse"])
    torch.manual_seed(0)
    flat = pose2mesh_net.get_model(17, mats).to(dev).eval()
    jr = torch.rand(17, 6890, generator=torch.Generator().manual_seed(3))
    jr = (jr / jr.sum(1, keepdim=True)).to(dev)
    people = torch.from_numpy(poses[:8]).to(dev)
    cam8 = c0[:8]

    def batched():
        flat.optimize_cam_param(people, perm_rev, 6890, jr, cam_init=cam8)

    def demo_style():
        for b in range(8):  # demo/run.py:149-189 per person: B = 1 network, then the Python loop
            with torch.no_grad():
                pose2d = postprocess.normalize_pose2d(people[b:b + 1])
                _, joints, _ = flat.predict_vertices_and_joints(pose2d, perm_rev, 6890, jr)
                target, _ = postprocess.crop_pose2d(people[b:b + 1])
            co.fit_camera(joints[0], target[0, :17], cam8[b])

    res["demo_8_people_ms"] = {"optimize_cam_param_batched": wall_ms(batched), "sequential_reference_style":
                               wall_ms(demo_style)}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
