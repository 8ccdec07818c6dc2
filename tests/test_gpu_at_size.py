"""GPU parity at the sizes BASELINE.json quotes (run on the B200 box with -m gpu).

configs[2]  B=256 forward+backward, SMPL-size hierarchy (V0 = 12288 ... 96), train-mode BatchNorm
configs[3]  MANO-size hierarchy (1088 ... 68), B=1024 forward+backward
configs[0]  demo/run.py single H36M pose (the reference's own input fixture) -> B=1 eval

The CPU oracle cannot run a 256-mesh TRAINING step of the SMPL-size network in test time (autograd keeps ~0.6 GB per
mesh), so the big batches are built from `n_distinct` distinct seeded poses repeated `copies` times
(b = c * n_distinct + i) with the targets repeated the same way.  Train-mode BatchNorm statistics, the loss and every
parameter gradient of the repeated batch equal those of the distinct batch (means over identical copies), and
dx[b] = dx_distinct[b % n_distinct] / copies, so the oracle only has to run the distinct poses — while the GPU path
runs the full batch: all tiles of all 148 persistent CTAs, the power-of-two fp16 gradient scaling over 3.1 M rows,
the TMEM accumulation of dW across every tile of a CTA, the fp64 BatchNorm sums.  Distinct meshes are interleaved
(period n_distinct), so a kernel that read another mesh's rows would be caught.
Tolerances (SURVEY.md §8d): outputs 1e-4 of max|y_ref| per mesh; gradients 1e-3 of the tensor's largest entry with
the ReLUs held open (BatchNorm bias +6), relative L2 1e-2 with live ReLUs (see test_gpu_parity.grad_close)."""
import numpy as np
import pytest
import torch

from helpers import CASES, load_npz
from test_gpu_parity import TOL_Y, dev, grad_close, per_mesh_rel_err

pytestmark = pytest.mark.gpu


def _hierarchy(name):
    from pose2mesh_release_b200 import graph as pg

    n, seed, levels, mano = CASES[name]
    face = pg.synthetic_sphere_faces(n, seed)
    if mano:
        _, graph_L, _, perm_rev = pg.build_coarse_graphs(face, 21, pg.MANO_SKELETON, pg.MANO_HORI_CONN, levels=levels)
    else:
        _, graph_L, _, perm_rev = pg.build_coarse_graphs(face, 17, pg.H36M_SKELETON, pg.H36M_FLIP_PAIRS, levels=levels)
    return graph_L, perm_rev, n, mano


def _train_step_parity(name, n_distinct, copies, open_relus, precision="fp16x3"):
    from oracle import meshnet_oracle as mo
    from pose2mesh_release_b200.meshnet import Pose2Mesh

    graph_L, _, _, mano = _hierarchy(name)
    n_joint = 21 if mano else 17
    torch.manual_seed(123)
    model = Pose2Mesh(5, 3, graph_L, joint_set="mano" if mano else "human36")
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    if open_relus:
        for k in sd:
            if k.startswith("bn.") and k.endswith(".bias"):
                sd[k].fill_(6.0)
        model.load_state_dict(sd)
    model = model.to(dev()).set_precision(precision).train()
    sd = {k: v.detach().cpu().clone() for k, v in sd.items()}
    laps = mo.laplacians_to_torch(graph_L)
    v0 = laps[0].shape[0]
    g = torch.Generator().manual_seed(41)
    xd = torch.randn(n_distinct, n_joint, 5, generator=g)
    td = torch.randn(n_distinct, v0, 3, generator=g)
    B = n_distinct * copies
    x = xd.repeat(copies, 1, 1).to(dev()).requires_grad_(True)
    tgt = td.repeat(copies, 1, 1).to(dev())
    y = model(x)
    loss = (y - tgt).abs().mean()
    del tgt

    sd_o = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "running" not in k else v.clone())
            for k, v in sd.items()}
    xo = xd.clone().requires_grad_(True)
    yo = mo.forward(sd_o, laps, xo, mano=mano, training=True)
    lo = (yo - td).abs().mean()
    lo.backward()
    # Both backward passes start from the same dL/dy, the oracle's sign(yo - td) / N.  The L1 loss has a kink at
    # y == tgt that open ReLUs do not hold open: of the B * V * 3 outputs, one can lie within the two fp32
    # implementations' difference of its target, flip sign, and move that mesh's dx by O(1e-3) of max |dx| (seen on
    # one host and not on another: |yo - td| = 4e-6 at 1 of 1.2 M entries, dx off by 1.8e-3 there, 7e-5 elsewhere).
    y.backward((torch.sign(yo.detach() - td).repeat(copies, 1, 1) / y.numel()).to(dev()))
    torch.cuda.synchronize()
    assert model._hier.kernel_status(torch.cuda.current_device()) == 0

    y_cpu = y.detach().cpu()
    assert y_cpu.shape == (B, v0, 3)
    assert per_mesh_rel_err(y_cpu, yo.detach().repeat(copies, 1, 1)) < TOL_Y
    assert abs(loss.item() - lo.item()) < 1e-5 * max(1.0, abs(lo.item()))
    ok, info = grad_close(x.grad * copies, xo.grad.repeat(copies, 1, 1), strict=open_relus)
    assert ok, ("dx", info)
    scale = max(float(v.grad.abs().max()) for v in sd_o.values() if v.requires_grad)
    worst = {}
    for k, p in model.named_parameters():
        ok, info = grad_close(p.grad, sd_o[k].grad, scale=1e-3 * scale, strict=open_relus)
        worst[k] = info
        assert ok, (k, info)
    info = model._hier.layer_info(torch.cuda.current_device())
    for k, v in model.state_dict().items():
        if k.endswith("running_mean"):
            # atol: 1e-5 of the (unit-scale) activations the mean is taken over — the oracle's own fp32 mean over
            # n_distinct * V rows is no more accurate than that
            np.testing.assert_allclose(v.cpu().numpy(), sd_o[k].numpy(), rtol=1e-4, atol=1e-5, err_msg=k)
        if k.endswith("running_var"):
            # running_var = 0.9 * 1 + 0.1 * biased_var * n / (n - 1) with n = rows of the batch: the repeated batch has
            # the same biased variance but n = B * V rows instead of n_distinct * V (matters on the 17-joint level)
            vl = info[int(k.split(".")[1])]["V"]
            n_o, n = n_distinct * vl, B * vl
            biased = (sd_o[k].numpy() - 0.9) / 0.1 * (n_o - 1) / n_o
            np.testing.assert_allclose(v.cpu().numpy(), 0.9 + 0.1 * biased * n / (n - 1), rtol=1e-4, atol=1e-5, err_msg=k)
        if k.endswith("num_batches_tracked"):
            assert int(v) == 1
    return worst


@pytest.mark.parametrize("open_relus", [True, False], ids=["open-relus-strict", "live-relus"])
def test_smpl_size_b256_train_step_against_oracle(open_relus):
    """BASELINE configs[2]: B=256 fwd+bwd on the SMPL-size hierarchy, 32 distinct poses x 8 (see the module docstring)."""
    _train_step_parity("smpl_like", 32, 8, open_relus)


@pytest.mark.parametrize("open_relus", [True, False], ids=["open-relus-strict", "live-relus"])
def test_mano_size_b1024_train_step_against_oracle(open_relus):
    """BASELINE configs[3]: MANO-size hierarchy, B=1024 fwd+bwd, 128 distinct poses x 8."""
    _train_step_parity("mano_like", 128, 8, open_relus)


@pytest.mark.parametrize("precision", ["fp32", "fp16x3"])
def test_demo_pose_b1_eval_against_oracle(precision):
    """BASELINE configs[0], the parity anchor: the reference's demo/h36m_joint_input.npy through the demo's own
    normalisation (demo/run.py:150-158, restated in oracle/demo_oracle.py and pinned to the reference's output in
    tests/golden/demo_pipeline.npz), combined with the reference PoseNet's 3-D lift for that pose
    (pose2mesh_net.py:18-19), then ONE mesh through MeshNet in eval mode on the SMPL-size hierarchy."""
    from oracle import demo_oracle as do
    from oracle import meshnet_oracle as mo
    from pose2mesh_release_b200.meshnet import Pose2Mesh

    z = load_npz("demo_pipeline.npz")
    pose2d = do.normalize_pose2d(load_npz("demo_input.npz")["joint_input"])
    np.testing.assert_allclose(pose2d, z["joint_img"][0], atol=1e-6)
    x = do.flat_pose2mesh_input(torch.from_numpy(pose2d)[None], torch.from_numpy(z["pose3d"][:1]))
    np.testing.assert_allclose(x.numpy(), z["pose_combine"][:1], atol=1e-6)
    graph_L, perm_rev, n_real, _ = _hierarchy("smpl_like")
    torch.manual_seed(123)
    model = Pose2Mesh(5, 3, graph_L, joint_set="human36")
    sd = mo.randomize_bn_({k: v.detach().clone() for k, v in model.state_dict().items()}, seed=7)
    model.load_state_dict(sd)
    model = model.to(dev()).set_precision(precision).eval()
    with torch.no_grad():
        y = model(x.to(dev()))                                     # B = 1 (demo/run.py:168-169)
        verts = model.forward_vertices(x.to(dev()), perm_rev, n_real)
        yo = mo.forward(sd, mo.laplacians_to_torch(graph_L), x, training=False)
    assert y.shape == (1, 12288, 3)
    assert per_mesh_rel_err(y, yo) < TOL_Y
    real = torch.as_tensor(np.asarray(perm_rev[:n_real]))
    assert per_mesh_rel_err(verts, yo[:, real]) < TOL_Y            # the 6890 vertices the demo keeps (run.py:170)


def test_data_parallel_two_gpus_matches_single_gpu():
    """The reference's multi-GPU mode is single-process nn.DataParallel (lib/core/base.py:108): worker threads, one
    replica per device, per-device native handles, gradients reduced onto device 0."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from test_gpu_parity import make_model

    model, mats, mano = make_model("mano_like", "fp16x3")
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    x = torch.randn(6, 21, 5, generator=torch.Generator().manual_seed(2)).to(dev())
    model.eval()
    with torch.no_grad():
        y1 = model(x)
    dp = torch.nn.DataParallel(model, device_ids=[0, 1])
    with torch.no_grad():
        y2 = dp(x)
    assert torch.cuda.current_device() == 0
    assert y2.device == x.device and per_mesh_rel_err(y2, y1) < 1e-6
    # training: per-replica BatchNorm like the reference; gradients flow back to the source parameters
    model.train()
    tgt = torch.randn(6, model.num_vertices, 3, device=dev())
    model.zero_grad()
    (dp(x) - tgt).abs().mean().backward()
    g_dp = {k: p.grad.clone() for k, p in model.named_parameters()}
    model.load_state_dict(sd)
    model.zero_grad()
    ya = model(x[:3])
    yb = model(x[3:])
    (torch.cat([ya, yb]) - tgt).abs().mean().backward()
    for k, p in model.named_parameters():
        ok, info = grad_close(g_dp[k], p.grad, scale=1e-6, strict=False)
        assert ok, (k, info)
