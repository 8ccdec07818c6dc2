"""TEST INFRASTRUCTURE ONLY — loader for the *unmodified* reference (hongsukchoi/Pose2Mesh_RELEASE).

Imports the reference's hot-path modules (lib/graph_utils.py, lib/coarsening.py,
lib/models/meshnet.py, lib/models/backbones/cheby_graph_conv.py) from /root/reference
in-process, with the three shims SURVEY.md §8(c) lists:

  1. stub ``core.config`` (the real one needs easydict and rmtree/mkdirs inside the
     read-only reference tree at import: lib/core/config.py:5-14,38);
  2. stub ``matplotlib`` / ``matplotlib.pyplot`` (lib/models/__init__.py:1-2 pulls
     posenet -> funcs_utils.py:12 -> pyplot; unused on this path);
  3. ``torch.Tensor.cuda`` -> identity while the reference runs on CPU
     (lib/models/meshnet.py:81 hard-codes .cuda()).

The reference tree is not part of this repository, so this module is used exclusively by
the fixture generators tests/golden/make_golden*.py; the tests compare with the fixtures
they wrote.  Nothing in the product path, the tests, smoke() or bench.py imports it.
"""
import contextlib
import os
import sys
import types

REF_ROOT = os.environ.get("P2M_REFERENCE_ROOT", "/root/reference")


def available() -> bool:
    return os.path.isdir(os.path.join(REF_ROOT, "lib", "models"))


class _Cfg:
    class DATASET:
        target_joint_set = "human36"

    class MODEL:
        posenet_pretrained = False
        posenet_path = ""
        input_shape = (384, 288)   # lib/core/config.py:52


_loaded = None


def load(target_joint_set: str = "human36"):
    """Return (graph_utils, coarsening, meshnet, cheby_graph_conv) reference modules."""
    global _loaded
    if not available():
        raise RuntimeError(f"reference tree not found at {REF_ROOT}")
    _Cfg.DATASET.target_joint_set = target_joint_set
    if _loaded is not None:
        return _loaded
    core = types.ModuleType("core")
    core.__path__ = []
    config = types.ModuleType("core.config")
    config.cfg = _Cfg
    core.config = config
    sys.modules.setdefault("core", core)
    sys.modules.setdefault("core.config", config)
    if "matplotlib" not in sys.modules:
        mpl = types.ModuleType("matplotlib")
        plt = types.ModuleType("matplotlib.pyplot")
        mpl.pyplot = plt
        mpl.use = lambda *a, **k: None
        sys.modules["matplotlib"] = mpl
        sys.modules["matplotlib.pyplot"] = plt
    lib = os.path.join(REF_ROOT, "lib")
    if lib not in sys.path:
        sys.path.insert(0, lib)
    import warnings

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        import coarsening  # noqa: E402  (reference module)
        import graph_utils  # noqa: E402
        from models import meshnet  # noqa: E402
        from models.backbones import cheby_graph_conv  # noqa: E402
    _loaded = (graph_utils, coarsening, meshnet, cheby_graph_conv)
    return _loaded


@contextlib.contextmanager
def cpu_cuda_noop():
    """Make Tensor.cuda() / Module.cuda() identities so meshnet.py:81 runs on CPU."""
    import torch

    old = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self
    try:
        yield
    finally:
        torch.Tensor.cuda = old
