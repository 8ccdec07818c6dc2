"""The demo's camera fit without a GPU (SURVEY.md §8 row f5): the CPU oracle (oracle/camera_oracle.py) against the
outputs of the unmodified reference (tests/golden/camera_fit.npz), the OptimzeCamLayer drop-in's surface, and the
native entry points refusing CPU tensors."""
import numpy as np
import pytest
import torch

from helpers import load_npz


def _cam(z, k):
    return torch.from_numpy(z[f"fit_cam_{k}"])


def test_crop_target_oracle_matches_reference_golden():
    from oracle import camera_oracle as co

    z = load_npz("camera_fit.npz")
    for i, (inp, is_int) in enumerate(zip(z["crop_input"], z["crop_input_is_int"])):
        tgt, bbox = co.crop_target(inp.astype(np.int64) if is_int else inp)
        np.testing.assert_array_equal(bbox, z["crop_bbox"][i])
        np.testing.assert_allclose(tgt, z["crop_target"][i], rtol=0, atol=1e-4)


def test_fit_oracle_matches_reference_golden():
    """The per-person loop on a few cases (every recorded step), the batched restatement on all of them: both follow
    the reference's fp32 trajectory."""
    from oracle import camera_oracle as co

    z = load_npz("camera_fit.npz")
    j3, tgt, c0 = (torch.from_numpy(z[k]) for k in ("fit_joints3d", "crop_target", "fit_cam_init"))
    for b in (0, 1, 17):
        cam, loss, snaps = co.fit_camera(j3[b], tgt[b], c0[b], record=(1, 10, 50))
        for k in (1, 10, 50):
            torch.testing.assert_close(snaps[k], _cam(z, k)[b], rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(co.project(j3[b:b + 1], cam[None]), co.project(j3[b:b + 1], _cam(z, 1500)[b:b + 1]),
                                   rtol=0, atol=0.05)
        assert abs(loss - z["fit_loss"][b]) <= 2e-3 * z["fit_loss"][b]
    for k in (10, 1500):
        cam, loss = co.fit_cameras_batched(j3, tgt, c0, iters=k)
        if k < 1500:
            torch.testing.assert_close(cam, _cam(z, k), rtol=1e-5, atol=1e-6)
        else:
            np.testing.assert_allclose(loss.numpy(), z["fit_loss"], rtol=2e-3)


def test_cam_layer_matches_reference_surface():
    from pose2mesh_release_b200 import project_net

    z = load_npz("camera_fit.npz")
    for s, ref in zip(z["init_seeds"], z["init_cam"]):
        torch.manual_seed(int(s))
        layer = project_net.get_model(500)
        assert list(layer.state_dict()) == ["cam_param"] and layer.cam_param.shape == (1, 3)
        assert layer.img_res == 250
        np.testing.assert_array_equal(layer.cam_param.detach()[0].numpy(), ref)
    torch.manual_seed(int(z["fwd_seed"]))
    layer = project_net.get_model(500)
    with torch.no_grad():
        out = layer(torch.from_numpy(z["fwd_in"]))
    np.testing.assert_array_equal(out.numpy(), z["fwd_out"])


def test_convert_crop_cam_matches_demo_formula():
    from pose2mesh_release_b200 import project_net

    cam = torch.tensor([[0.9, 0.1, -0.05], [1.1, -0.2, 0.3]], dtype=torch.float64)
    bbox = torch.tensor([[55.9, 78.9, 651.25, 651.25], [300.0, 200.0, 500.0, 500.0]], dtype=torch.float64)
    got = project_net.convert_crop_cam_to_orig_img(cam, bbox, 1280, 720).numpy()
    c, b = cam.numpy(), bbox.numpy()
    h = b[:, 3]
    sx, sy = c[:, 0] * h / 1280, c[:, 0] * h / 720
    ref = np.stack([sx, sy, (b[:, 0] + b[:, 2] / 2 - 640) / 640 / sx + c[:, 1],
                    (b[:, 1] + h / 2 - 360) / 360 / sy + c[:, 2]], axis=1)
    np.testing.assert_allclose(got, ref, rtol=1e-12)


def test_native_fit_refuses_cpu_tensors():
    from pose2mesh_release_b200 import project_net

    p, t, c = torch.zeros(2, 17, 3), torch.zeros(2, 17, 2), torch.rand(2, 3)
    with pytest.raises(RuntimeError, match="CUDA"):
        project_net.fit_camera(p, t, 500, c)
    with pytest.raises(RuntimeError, match="CUDA"):
        project_net.get_model(500).fit(p[:1], t[:1])
