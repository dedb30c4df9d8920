"""Golden vectors at the BENCHMARKED shapes, generated from the UNMODIFIED reference.

Run in the build container only (the GPU box has no /root/reference):

    python tests/golden/make_golden_big.py c3        # 150 x 360 x 640, full loop (~17 GB RSS)
    python tests/golden/make_golden_big.py c2        # 30 x 360 x 480, flow + tracks
    python tests/golden/make_golden_big.py c4slice   # 24 x 720 x 1280, flow only
    python tests/golden/make_golden_big.py c3 3 --f64   # the same in float64 (arbiter, ~35 GB RSS)

The inputs are NOT stored: they are `bench.synthetic_inputs(f, h, w, seed)` and
`bench.synthetic_track_arrays(f, seed=seed)` (torch's seeded CPU generator), which the GPU
tests regenerate; the fixture keeps the reference's outputs in reduced form -- loss parts,
all poses, the focal length, and for every full-size gradient / parameter tensor its per-frame
L2 norms plus a strided subsample (every STRIDES[case]-th element: multiples of 61, so that the
samples wander through the columns, chosen to keep every fixture under 1 MB).  The Lightning
shell is restated as in make_golden.py (model_wrapper_overfit.py:51-73, 104-105); the softmin point indices are injected by patching
torch.randperm (SURVEY A.8 item 1): the first `softmin_points` entries of
torch.randperm(h * w, generator=manual_seed(3)).
"""
from __future__ import annotations

import os
import sys
import time
from pathlib import Path

import numpy as np
import torch

REF = "/root/reference"
OUT = Path(__file__).resolve().parent
ROOT = OUT.parent.parent
sys.path.insert(0, str(ROOT))
STRIDES = {"c2": 122, "c3": 732, "c4slice": 488}
START_STEP = 50  # bench.START_STEP: tracking loss on (>= 50), softmin stage (< 1000)


def reduced(name, t):
    """Per-frame L2 norms (float64) and a strided subsample of a (frames, h, w) tensor."""
    t = t.detach()
    return {f"{name}_norms": t.double().flatten(1).norm(dim=1).numpy(),
            f"{name}_sub": t.flatten()[::STRIDE].float().numpy()}


def main():
    which = sys.argv[1] if len(sys.argv) > 1 else "c3"
    steps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    f64 = "--f64" in sys.argv
    sys.path.insert(0, REF)
    os.environ["PYTHONDONTWRITEBYTECODE"] = "1"
    sys.dont_write_bytecode = True
    torch.set_num_threads(os.cpu_count() or 8)
    import bench
    cases = {
        # name: (f, h, w, intrinsics, tracking, softmin points)
        "c3": (150, 360, 640, "softmin", True, 8192),
        "c2": (30, 360, 480, "softmin", True, 8192),
        "c4slice": (24, 720, 1280, "regressed", False, 0),
    }
    f, h, w, intr, tracking, npts = cases[which]
    seed = 0
    # the inputs are the float32 values the GPU tests regenerate (drawn BEFORE any dtype games)
    inp32 = bench.synthetic_inputs(f, h, w, seed=seed)
    trk32 = bench.synthetic_track_arrays(f, seed=seed) if tracking else None
    perm = torch.randperm(h * w, generator=torch.Generator().manual_seed(3))
    if f64:  # the float64 arbiter: rebind the NAME torch.float32 before importing the reference, which
        # hard-codes it in a dozen places (same recipe as make_golden.py; SURVEY A.9)
        torch.float32 = torch.float64
        torch.set_default_dtype(torch.float64)
    dtype = torch.float64 if f64 else torch.float32
    from flowmap.dataset.types import Batch
    from flowmap.flow.flow_predictor import Flows
    from flowmap.loss import get_losses
    from flowmap.loss.loss_flow import LossFlowCfg
    from flowmap.loss.loss_tracking import LossTrackingCfg
    from flowmap.loss.mapping.mapping_huber import MappingHuberCfg
    from flowmap.model.backbone.backbone_explicit_depth import BackboneExplicitDepthCfg
    from flowmap.model.extrinsics.extrinsics_procrustes import ExtrinsicsProcrustesCfg
    from flowmap.model.intrinsics.intrinsics_regressed import IntrinsicsRegressedCfg
    from flowmap.model.intrinsics.intrinsics_softmin import IntrinsicsSoftminCfg, RegressionCfg
    from flowmap.model.model import Model, ModelCfg
    from flowmap.tracking.track_predictor import Tracks

    global STRIDE
    STRIDE = STRIDES[which]
    seed = 0
    inp = {k: v.to(dtype) for k, v in inp32.items()}
    if intr == "softmin":
        icfg = IntrinsicsSoftminCfg("softmin", npts, 0.5, 2.0, 60, RegressionCfg(1000, 100))
    else:
        icfg = IntrinsicsRegressedCfg("regressed", 0.85)
    mcfg = ModelCfg(BackboneExplicitDepthCfg("explicit_depth", 0.1, 100.0), icfg,
                    ExtrinsicsProcrustesCfg("procrustes", None, False), True)
    model = Model(mcfg, f, (h, w))
    with torch.no_grad():
        model.backbone.depth.copy_(inp["depth"])
        model.backbone.weights.copy_(inp["wparam"])
    huber = MappingHuberCfg("huber", 0.01)
    lcfgs = [LossFlowCfg(0, 1000.0, "flow", huber)]
    tracks = None
    if tracking:
        lcfgs.append(LossTrackingCfg(50, 100.0, "tracking", huber))
        tracks = [Tracks(xy.to(dtype), vis, s) for xy, vis, s in trk32]
    losses = get_losses(lcfgs)
    batch = Batch(torch.zeros((1, 1, 1, 1, 1), dtype=dtype).expand(1, f, 3, h, w), torch.arange(f)[None], ["s"], ["d"])
    flows = Flows(inp["fwd"], inp["bwd"], inp["fmask"], inp["bmask"])

    real_randperm = torch.randperm
    torch.randperm = lambda n, **kw: perm
    opt = torch.optim.Adam(model.parameters(), lr=3e-5)  # model_wrapper_overfit.py:104-105
    rec = {"loss": [], "loss_flow": [], "loss_tracking": [], "extrinsics": [], "fx": []}
    out_arrays = {}
    try:
        for s in range(steps):
            t0 = time.time()
            opt.zero_grad()
            gs = START_STEP + s
            out = model(batch, flows, gs)
            parts = [l.forward(batch, flows, tracks, out, gs) for l in losses]
            total = sum(parts)
            total.backward()
            if s == 0:  # gradients of the first step, before Adam touches anything
                out_arrays.update(reduced("g_depth", model.backbone.depth.grad))
                out_arrays.update(reduced("g_wparam", model.backbone.weights.grad))
                fl = getattr(model.intrinsics, "focal_length", None)
                if fl is not None and fl.grad is not None:
                    out_arrays["g_focal"] = fl.grad.numpy()
            opt.step()
            rec["loss"].append(float(total))
            rec["loss_flow"].append(float(parts[0]))
            rec["loss_tracking"].append(float(parts[1]) if tracking else 0.0)
            rec["extrinsics"].append(out.extrinsics.detach()[0].numpy().copy())
            rec["fx"].append(float(out.intrinsics[0, 0, 0, 0]))
            print(f"{which} step {s}: loss {float(total):.6f} ({time.time() - t0:.1f} s)", flush=True)
    finally:
        torch.randperm = real_randperm
    out_arrays.update(reduced("depth_final", model.backbone.depth))
    out_arrays.update(reduced("wparam_final", model.backbone.weights))
    np.savez_compressed(
        OUT / f"big_{which}{'_f64' if f64 else ''}.npz", frames=f, height=h, width=w, seed=seed, stride=STRIDE,
        start_step=START_STEP, softmin_indices=perm[:npts].numpy() if npts else np.zeros(0, np.int64),
        loss=np.array(rec["loss"]), loss_flow=np.array(rec["loss_flow"]),
        loss_tracking=np.array(rec["loss_tracking"]), extrinsics=np.stack(rec["extrinsics"]),
        fx=np.array(rec["fx"]), **out_arrays)
    out_path = OUT / f"big_{which}{'_f64' if f64 else ''}.npz"
    print("wrote", out_path, out_path.stat().st_size / 1e6, "MB")


if __name__ == "__main__":
    main()
