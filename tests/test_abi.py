"""The C-ABI library loads on a CPU-only box and exports every symbol the header declares."""
import ctypes
import re

from conftest import ROOT


def declared_symbols():
    text = (ROOT / "include" / "flowmap_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(fm_[a-z0-9_]+)\s*\(", text)))


def test_library_builds_and_exports_header_symbols():
    from flowmap_b200.build import build
    from flowmap_b200 import _lib
    so = build()
    handle = ctypes.CDLL(str(so))
    names = declared_symbols()
    assert len(names) >= 10
    for name in names:
        assert hasattr(handle, name), f"{name} declared in the header but not exported"
        assert name in _lib.SIGNATURES, f"{name} has no ctypes signature"
    assert set(_lib.SIGNATURES) == set(names)
    assert _lib.lib().fm_version() >= 100
    # pure host-side query works without a GPU
    assert _lib.lib().fm_workspace_bytes(1, 150, 360, 640) > 0
    assert _lib.lib().fm_workspace_bytes(1, 1, 8, 8) == 0


def test_product_has_no_cpu_path():
    import pytest
    import torch
    from flowmap_b200 import ops
    d = torch.zeros(1, 2, 4, 4)
    with pytest.raises(ValueError, match="CUDA"):
        ops.procrustes_poses(d, None, torch.zeros(1, 2, 4), torch.zeros(1, 1, 4, 4, 2))


def test_package_does_not_import_oracle():
    import subprocess, sys
    code = ("import sys, flowmap_b200, flowmap_b200.model, flowmap_b200.loss, flowmap_b200.overfit;"
            "bad=[m for m in sys.modules if m.startswith('oracle')]; assert not bad, bad")
    subprocess.check_call([sys.executable, "-c", code], cwd=str(ROOT))


PROJECTION_NAMES = ("sample_image_grid", "unproject", "project", "reproject_points", "compute_forward_flow",
                    "compute_backward_flow", "get_extrinsics", "align_surfaces")

# The parts of the reference's `flowmap` package that install() touches, reduced to their names:
# the registries with the reference's keys, the projection / Procrustes helpers, the modules that
# import helpers by name, and FlowPredictor's static methods.  flowmap.export.colmap is absent,
# as it is wherever `plyfile` is not installed.
STAND_IN = {
    "flowmap/__init__.py": "",
    "flowmap/model/__init__.py": "",
    "flowmap/model/projection.py": "".join(f"def {n}(*args): pass\n" for n in PROJECTION_NAMES),
    "flowmap/model/procrustes.py": "def align_rigid(*args): pass\n",
    "flowmap/model/model.py": "from .projection import sample_image_grid, unproject\nclass Model: pass\n",
    "flowmap/model/backbone/__init__.py": "class Midas: pass\nclass ExplicitDepth: pass\n"
                                          "BACKBONES = {'explicit_depth': ExplicitDepth, 'midas': Midas}\n",
    "flowmap/model/intrinsics/__init__.py": "INTRINSICS = {'ground_truth': 0, 'regressed': 0, 'softmin': 0}\n",
    "flowmap/model/intrinsics/intrinsics_softmin.py":
        "from ..projection import align_surfaces, compute_backward_flow, sample_image_grid, unproject\n",
    "flowmap/model/extrinsics/__init__.py": "EXTRINSICS = {'procrustes': 0, 'regressed': 0}\n",
    "flowmap/model/extrinsics/extrinsics_regressed.py": "from ..projection import get_extrinsics\n",
    "flowmap/loss/__init__.py": "LOSSES = {'flow': 0, 'tracking': 0}\n",
    "flowmap/flow/__init__.py": "",
    "flowmap/flow/flow_predictor.py": "class FlowPredictor:\n"
                                      "    rescale_flow = rescale_mask = compute_consistency_mask = staticmethod(id)\n",
}

# What install() reported replacing when run against the unmodified reference package.
REPLACED_IN_REFERENCE = [
    "flowmap.flow.flow_predictor.FlowPredictor.compute_consistency_mask",
    "flowmap.flow.flow_predictor.FlowPredictor.rescale_flow",
    "flowmap.flow.flow_predictor.FlowPredictor.rescale_mask",
    "flowmap.loss.LOSSES[flow]", "flowmap.loss.LOSSES[tracking]",
    "flowmap.model.extrinsics.EXTRINSICS[procrustes]", "flowmap.model.extrinsics.EXTRINSICS[regressed]",
    "flowmap.model.intrinsics.INTRINSICS[ground_truth]", "flowmap.model.intrinsics.INTRINSICS[regressed]",
    "flowmap.model.intrinsics.INTRINSICS[softmin]",
    "flowmap.model.model.Model", "flowmap.model.procrustes.align_rigid",
    *(f"flowmap.model.projection.{n}" for n in sorted(PROJECTION_NAMES)),
]


def test_install_patches_reference_registries(tmp_path):
    """flowmap_b200.install() against a stand-in for the reference's package layout; the reference's
    config objects are given as plain namespaces carrying the reference's field names."""
    import subprocess, sys
    from conftest import ROOT
    for rel, text in STAND_IN.items():
        (tmp_path / rel).parent.mkdir(parents=True, exist_ok=True)
        (tmp_path / rel).write_text(text)
    code = (
        f"import sys; sys.path.insert(0, {str(tmp_path)!r}); sys.dont_write_bytecode = True\n"
        "from types import SimpleNamespace as ns\n"
        "import flowmap_b200, flowmap.model.model as rm, flowmap.loss as rl, flowmap.model.backbone as rb\n"
        "import flowmap.model.intrinsics as ri, flowmap.model.extrinsics as re_\n"
        "import flowmap.model.projection as rp, flowmap.model.procrustes as rpr\n"
        "import flowmap.model.intrinsics.intrinsics_softmin as rsoft, flowmap.model.extrinsics.extrinsics_regressed as rreg\n"
        "midas = rb.BACKBONES['midas']\n"
        "rep = flowmap_b200.install()\n"
        f"assert sorted(rep) == {REPLACED_IN_REFERENCE!r}, sorted(rep)\n"
        "from flowmap_b200 import model as mm, projection as mp, procrustes as mpr, flow as fl\n"
        "from flowmap_b200.loss import LossFlow, LossTracking\n"
        "assert rm.Model is mm.Model and rl.LOSSES['flow'] is LossFlow and rl.LOSSES['tracking'] is LossTracking\n"
        "assert all(ri.INTRINSICS[k] is mm.INTRINSICS[k] for k in ri.INTRINSICS)\n"
        "assert all(re_.EXTRINSICS[k] is mm.EXTRINSICS[k] for k in re_.EXTRINSICS)\n"
        "assert mm.BACKBONES['midas'] is midas and mm.BACKBONES['explicit_depth'] is not rb.BACKBONES['explicit_depth']\n"
        "assert rpr.align_rigid is mpr.align_rigid\n"
        "for mod in (rp, rm, rsoft, rreg):\n"
        "    for n in dir(mod):\n"
        "        if not n.startswith('_') and n != 'Model':\n"
        "            assert getattr(mod, n) is getattr(mp, n), (mod.__name__, n)\n"
        "cfg = ns(backbone=ns(name='explicit_depth', initial_depth=0.1, weight_sensitivity=100.0),\n"
        "         intrinsics=ns(name='softmin', num_procrustes_points=8192, min_focal_length=0.5, max_focal_length=2.0,\n"
        "                       num_candidates=60, regression=ns(after_step=1000, window=100)),\n"
        "         extrinsics=ns(name='procrustes', num_points=None, randomize_points=False),\n"
        "         use_correspondence_weights=True)\n"
        "m = rm.Model(cfg, 4, (8, 12))\n"
        "names = sorted(n for n, _ in m.named_parameters())\n"
        "assert names == ['backbone.depth', 'backbone.weights', 'intrinsics.intrinsics_regressed.focal_length'], names\n"
        "loss_cfg = ns(enable_after=0, weight=1000.0, name='flow', mapping=ns(name='huber', delta=0.01))\n"
        "assert type(rl.LOSSES[loss_cfg.name](loss_cfg)) is LossFlow\n"
        "from flowmap.flow.flow_predictor import FlowPredictor\n"
        "assert FlowPredictor.rescale_flow is fl.rescale_flow and FlowPredictor.rescale_mask is fl.rescale_mask\n"
        "assert FlowPredictor.compute_consistency_mask is fl.compute_consistency_mask\n")
    subprocess.check_call([sys.executable, "-c", code], cwd=str(ROOT))
