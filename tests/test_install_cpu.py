"""install() / uninstall(): the rebinding overlay over an UNMODIFIED reference checkout (SURVEY.md §8b).
CPU-only and self-contained: the reference's modules are stood in for by stubs registered under the names install()
imports, binding their names the way the reference's modules do; what the reference's classes produce (state_dict
keys, shapes and seeded initial values) comes from the golden fixtures made by the unmodified reference
(meshnet_smpl_small.npz, posenet_state_dict.npz)."""
import importlib
import sys
import types

import numpy as np
import pytest
import torch

from helpers import graph_from_fixture, load_npz

_LAYOUT = ("core", "core.config", "graph_utils", "models", "models.backbones", "models.backbones.cheby_graph_conv",
           "models.meshnet", "models.posenet", "models.pose2mesh_net")


def _reference_layout():
    """Stub modules with the reference's names and bindings; its functions and classes refuse to run, so a test that
    reached one of them after install() would fail."""
    mods = {name: types.ModuleType(name) for name in _LAYOUT}
    for pkg in ("core", "models", "models.backbones"):
        mods[pkg].__path__ = []
    for name in _LAYOUT:
        parent, _, leaf = name.rpartition(".")
        if parent:
            setattr(mods[parent], leaf, mods[name])

    def original(name):
        def fn(*args, **kwargs):
            raise AssertionError(f"the reference's {name} ran although install() rebound it")
        fn.__name__ = name
        return fn

    mods["core.config"].cfg = types.SimpleNamespace(DATASET=types.SimpleNamespace(target_joint_set="human36"),
                                                    MODEL=types.SimpleNamespace(posenet_pretrained=False))
    gu, conv, meshnet, posenet, flat = (mods[n] for n in ("graph_utils", "models.backbones.cheby_graph_conv",
                                                         "models.meshnet", "models.posenet", "models.pose2mesh_net"))
    gu.build_coarse_graphs = original("build_coarse_graphs")
    conv.graph_conv_cheby = original("graph_conv_cheby")
    meshnet.graph_utils = gu
    meshnet.graph_conv_cheby = conv.graph_conv_cheby        # meshnet.py:9 imports the function by name
    meshnet.Pose2Mesh, meshnet.get_model = type("Pose2Mesh", (torch.nn.Module,), {}), original("meshnet.get_model")
    posenet.LinearModel, posenet.get_model = type("LinearModel", (torch.nn.Module,), {}), original("posenet.get_model")
    flat.meshnet, flat.posenet = meshnet, posenet

    def get_model(num_joint, graph_L):
        """pose2mesh_net.py:8-14,24-27: FlatPose2Mesh looks both halves up on the module objects when it is built."""
        model = torch.nn.Module()
        model.num_joint = num_joint
        model.pose_lifter = flat.posenet.get_model(num_joint, hid_dim=4096, num_layer=2, p_dropout=0.5,
                                                   pretrained=mods["core.config"].cfg.MODEL.posenet_pretrained)
        model.pose2mesh = flat.meshnet.get_model(num_joint_input_chan=2 + 3, num_mesh_output_chan=3, graph_L=graph_L)
        return model

    flat.get_model = get_model
    return mods


@pytest.fixture()
def reference():
    saved = {name: sys.modules.get(name) for name in _LAYOUT}
    mods = _reference_layout()
    sys.modules.update(mods)
    import pose2mesh_release_b200.install as inst

    try:
        yield mods["graph_utils"], mods["models.meshnet"], mods["models.backbones.cheby_graph_conv"], inst
    finally:
        inst.uninstall()
        for name, mod in saved.items():
            if mod is None:
                sys.modules.pop(name, None)
            else:
                sys.modules[name] = mod


def test_install_rebinds_every_holder_and_uninstall_restores(reference):
    gu, ref_meshnet, ref_conv, inst = reference
    import pose2mesh_release_b200 as p2m
    from pose2mesh_release_b200 import cheby_graph_conv as my_conv
    from pose2mesh_release_b200 import graph as my_graph

    orig = (ref_meshnet.Pose2Mesh, ref_meshnet.get_model, ref_conv.graph_conv_cheby, gu.build_coarse_graphs)
    # a module imported BEFORE install() that holds its own binding, like the reference's datasets and demo/run.py
    # (`from graph_utils import build_coarse_graphs`, data/Human36M/dataset.py:13, demo/run.py:18)
    holder = type(sys)("early_holder")
    holder.build_coarse_graphs = gu.build_coarse_graphs
    holder.graph_conv_cheby = ref_conv.graph_conv_cheby
    sys.modules["early_holder"] = holder
    try:
        inst.install()
        assert ref_meshnet.Pose2Mesh is p2m.Pose2Mesh and ref_meshnet.get_model is p2m.get_model
        assert ref_conv.graph_conv_cheby is my_conv.graph_conv_cheby
        assert ref_meshnet.graph_conv_cheby is my_conv.graph_conv_cheby     # meshnet.py:9 imported the name
        assert gu.build_coarse_graphs is my_graph.build_coarse_graphs
        assert holder.build_coarse_graphs is my_graph.build_coarse_graphs
        assert holder.graph_conv_cheby is my_conv.graph_conv_cheby
        inst.install()                                                       # idempotent
        inst.uninstall()
        assert (ref_meshnet.Pose2Mesh, ref_meshnet.get_model, ref_conv.graph_conv_cheby, gu.build_coarse_graphs) == orig
        assert holder.build_coarse_graphs is orig[3] and holder.graph_conv_cheby is orig[2]
    finally:
        sys.modules.pop("early_holder", None)


def test_flat_pose2mesh_builds_the_b200_meshnet(reference):
    """The reference's own wrapper (lib/models/pose2mesh_net.py:5,14 -> meshnet.get_model) picks the overlay up,
    with the reference's state_dict keys under the `pose2mesh.` prefix."""
    gu, ref_meshnet, ref_conv, inst = reference
    import pose2mesh_release_b200 as p2m

    mats, _ = graph_from_fixture("smpl_small")
    z = load_npz("meshnet_smpl_small.npz")                                    # the reference's Pose2Mesh on these graphs
    ref_keys = [str(k) for k in z["keys"]]
    inst.install()
    pose2mesh_net = importlib.import_module("models.pose2mesh_net")
    flat = pose2mesh_net.get_model(17, [m.copy() for m in mats])
    assert isinstance(flat.pose2mesh, p2m.Pose2Mesh)
    from pose2mesh_release_b200 import posenet as my_posenet

    assert isinstance(flat.pose_lifter, my_posenet.LinearModel)               # the front half is rebound as well
    got = sorted(k[len("pose2mesh."):] for k in flat.state_dict() if k.startswith("pose2mesh."))
    assert got == ref_keys
    ref_sd = {k: torch.zeros(tuple(int(s) for s in z["shape/" + k])) for k in ref_keys}
    flat.pose2mesh.load_state_dict(ref_sd)                                    # reference checkpoints load unchanged
    # drop-in users get the tensor-core path without touching the module (P2M_PRECISION overrides)
    from pose2mesh_release_b200 import _lib

    assert flat.pose2mesh._hier.precision == _lib.default_precision() == _lib.P2M_PREC_FP16X3_TC
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="CUDA"):
            flat.pose2mesh(torch.zeros(1, 17, 5))


def test_precision_env_override(monkeypatch):
    from pose2mesh_release_b200 import _lib

    monkeypatch.setenv("P2M_PRECISION", "fp32")
    assert _lib.default_precision() == _lib.P2M_PREC_FP32_SIMT
    monkeypatch.setenv("P2M_PRECISION", "bf16")
    with pytest.raises(RuntimeError, match="P2M_PRECISION"):
        _lib.default_precision()


def test_posenet_mirror_has_the_reference_state_dict():
    """models.posenet.LinearModel (lib/models/posenet.py:41-72) and the B200 mirror: same keys, shapes and — under the
    same seed — the same initial values, so PoseNet checkpoints load unchanged."""
    from pose2mesh_release_b200 import pose2mesh_net as my_flat
    from pose2mesh_release_b200 import posenet as my_posenet

    z = load_npz("posenet_state_dict.npz")          # reference get_model(17, 64, 2, 0.5) under torch.manual_seed(5)
    torch.manual_seed(5)
    mine = my_posenet.get_model(17, hid_dim=64, num_layer=2, p_dropout=0.5, pretrained=False)
    ms = mine.state_dict()
    assert list(ms.keys()) == [str(k) for k in z["keys"]]
    for k, v in ms.items():
        ref = torch.from_numpy(np.asarray(z["sd/" + k]))
        assert ref.shape == v.shape and torch.equal(ref, v), k
    mats, _ = graph_from_fixture("smpl_small")
    flat = my_flat.get_model(17, [m.copy() for m in mats])
    assert {k.split(".")[0] for k in flat.state_dict()} == {"pose_lifter", "pose2mesh"}   # pose2mesh_net.py:13-14
