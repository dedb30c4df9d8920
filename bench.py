#!/usr/bin/env python
"""Benchmark of the FlowMap optimisation hot path on B200 (contract: DESIGN.md section 6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--mode scenes|pairs]
                    [--dump-outputs DIR]

One "step" = one full overfit iteration at BASELINE config 3 (150 x 360 x 640, synthetic):
explicit-depth backbone, all-pixel Procrustes, softmin intrinsics (60-candidate sweep), flow
loss + tracking loss (30 segments x 1225 tracks), backward, Adam -- what
flowmap/model/model_wrapper_overfit.py:51-73,104-105 runs per iteration with the reference's
default losses/intrinsics and `+experiment=ablation_explicit_depth`.
N > 1 (default --mode scenes, BASELINE config 5): one independent scene per GPU, no data-path
collective.  --mode pairs (config 4 style): flow-loss-only run of ONE long video whose frame
pairs are sharded across ranks, one all-reduce per step.  Prints ONE JSON line on rank 0.
--dump-outputs DIR writes what the last timed step computed on rank 0 as DIR/<name>.npy (see
dump_outputs); the inputs are seeded, so two builds can be compared output for output.
The benchmark writes nothing into the source tree.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True  # the tree may be read-only; leave no __pycache__ in it

F_, H_, W_ = 150, 360, 640  # BASELINE.json configs[2] ("Tanks&Temples-shape")
START_STEP = 50             # tracking loss enabled (>= 50), softmin stage (< 1000)
WORKLOAD = ("C3 150x360x640 synthetic (iid N(0,0.01^2) flows, U(0,1) masks, 30 track segments x "
            "1225 uniform tracks), explicit_depth backbone, all-pixel Procrustes, softmin "
            "intrinsics (60 candidates x 8192 points), flow + tracking loss (Huber), full overfit "
            "step = Model.forward + losses + backward + Adam, global_step >= 50")
METRIC = "overfit iters/sec at 150x360x640 (149 frame pairs per iteration)"


# ------------------------------------------------------------------------------ inputs
def synthetic_inputs(f, h, w, seed=0):
    """SURVEY 8(d) "throughput set": depth 0.1+0.05 U, weight logits N(0,.01), flows
    N(0, .01^2) in normalised units, masks U(0,1).  CPU float32 tensors."""
    g = torch.Generator().manual_seed(seed)
    p = f - 1
    return {
        "depth": 0.1 + 0.05 * torch.rand(f, h, w, generator=g),
        "wparam": 0.01 * torch.randn(p, h, w, generator=g),
        "fwd": 0.01 * torch.randn(1, p, h, w, 2, generator=g),
        "bwd": 0.01 * torch.randn(1, p, h, w, 2, generator=g),
        "fmask": torch.rand(1, p, h, w, generator=g),
        "bmask": torch.rand(1, p, h, w, generator=g),
    }


def synthetic_track_arrays(f, n_points=1225, interval=5, radius=20, seed=0):
    """Segment layout of flowmap/tracking/__init__.py:49-70 (one segment every `interval`
    frames covering [mid - radius, mid + radius]); xy ~ U(0,1)^2, visibility ~ Bernoulli(.7).
    Returns a list of (xy (1, fs, n, 2), vis (1, fs, n) bool, start_frame)."""
    g = torch.Generator().manual_seed(seed + 1)
    out = []
    for mid in range(0, f, interval):
        lo, hi = max(0, mid - radius), min(f, mid + radius + 1)
        out.append((torch.rand(1, hi - lo, n_points, 2, generator=g),
                    torch.rand(1, hi - lo, n_points, generator=g) < 0.7, lo))
    return out


def algorithmic_bytes(f, h, w):
    """SURVEY 8(d): 32 B per pair-pixel + 8 B per frame-pixel."""
    return h * w * (32 * (f - 1) + 8 * f)


DUMP_SAMPLE = 1 << 21  # elements kept of each per-pixel array (4 arrays x 8 MB)


def dump_outputs(out_dir, o, last):
    """Write what the last step of `o` computed, as float32 .npy files under `out_dir`: the total
    loss and relative poses it returned, the (fx, fy, cx, cy) it used, the focal-length gradient,
    and of the per-pixel arrays (updated depth and weight logits, their gradients; 138 MB each at
    the benchmark shape) the same fixed, seeded sample of elements in every run."""
    import numpy as np
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    loss, rt = last
    grads = o.gradients()
    arrays = {"loss": loss, "rt": rt, "intrinsics_k4": o.intrinsics_k4(), "g_focal": grads["focal"]}
    per_pixel = {"depth": o.model.backbone.depth, "weight_logits": o.model.backbone.weights,
                 "g_depth": grads["depth"], "g_weight_logits": grads["weights"]}
    picks = {}
    for name, t in per_pixel.items():
        flat = t.detach().reshape(-1)
        n = flat.numel()
        if n not in picks:
            g = torch.Generator().manual_seed(n)
            picks[n] = torch.randperm(n, generator=g)[:DUMP_SAMPLE].sort().values.to(flat.device)
        arrays[f"{name}_sample"] = flat[picks[n]]
    for name, t in arrays.items():
        np.save(out_dir / f"{name}.npy", t.detach().float().cpu().numpy())


# ------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi sampled every 20 ms in the background; samples are time-stamped so that the
    ones that fall inside the timed regions can be picked out afterwards."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.samples, self.proc, self.index, self.windows = [], None, index, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-i", str(self.index), "-lms", "20"], stdout=subprocess.PIPE,
                stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.time(), line.strip()))

    def window(self, t0, t1):
        self.windows.append((t0, t1))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        inside = [r for r in self.samples if any(a <= r[0] <= b for a, b in self.windows)]
        which = "timed regions"
        if len(inside) < 3:  # regions shorter than the sampling period
            inside, which = self.samples, "warm-up + timed regions + per-op timing (all under load)"
        sm, mx, reasons = [], None, set()
        for _, s in inside:
            parts = [x.strip() for x in s.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm), "window": which}


# ------------------------------------------------------------------------------ the reference itself
REF_DIR = ROOT / "baseline" / "_ref"


def reference_available():
    return (REF_DIR / "flowmap" / "model" / "model.py").exists()


def reference_runner(device, frames=F_, h=H_, w=W_, seed=0):
    """The UNMODIFIED reference (baseline/_ref, staged by baseline/install_ref.py) on `device`:
    flowmap.model.model.Model + flowmap.loss.get_losses driven as model_wrapper_overfit.py:51-73,
    104-105 does (Lightning / Hydra are not installed: only that shell is restated), with the
    values of config/overfit.yaml + experiment/ablation_explicit_depth.yaml on the bench workload.
    Returns step() -> float loss (one full overfit iteration incl. Adam)."""
    if str(REF_DIR) not in sys.path:
        sys.path.insert(0, str(REF_DIR))
    sys.dont_write_bytecode = True
    from flowmap.dataset.types import Batch as RBatch
    from flowmap.flow.flow_predictor import Flows as RFlows
    from flowmap.loss import get_losses as r_get_losses
    from flowmap.loss.loss_flow import LossFlowCfg as RLossFlowCfg
    from flowmap.loss.loss_tracking import LossTrackingCfg as RLossTrackingCfg
    from flowmap.loss.mapping.mapping_huber import MappingHuberCfg as RHuber
    from flowmap.model.backbone.backbone_explicit_depth import BackboneExplicitDepthCfg as RBackboneCfg
    from flowmap.model.extrinsics.extrinsics_procrustes import ExtrinsicsProcrustesCfg as RExtrCfg
    from flowmap.model.intrinsics.intrinsics_softmin import IntrinsicsSoftminCfg as RSoftminCfg
    from flowmap.model.intrinsics.intrinsics_softmin import RegressionCfg as RRegressionCfg
    from flowmap.model.model import Model as RModel
    from flowmap.model.model import ModelCfg as RModelCfg
    from flowmap.tracking.track_predictor import Tracks as RTracks

    inp = synthetic_inputs(frames, h, w, seed=seed)
    mcfg = RModelCfg(RBackboneCfg("explicit_depth", 0.1, 100.0),
                     RSoftminCfg("softmin", 8192, 0.5, 2.0, 60, RRegressionCfg(1000, 100)),
                     RExtrCfg("procrustes", None, False), True)
    model = RModel(mcfg, frames, (h, w))
    with torch.no_grad():
        model.backbone.depth.copy_(inp["depth"])
        model.backbone.weights.copy_(inp["wparam"])
    model.to(device)
    huber = RHuber("huber", 0.01)
    losses = r_get_losses([RLossFlowCfg(0, 1000.0, "flow", huber), RLossTrackingCfg(50, 100.0, "tracking", huber)])
    batch = RBatch(torch.zeros((1, 1, 1, 1, 1), device=device).expand(1, frames, 3, h, w),
                   torch.arange(frames, device=device)[None], ["synthetic"], ["synthetic"])
    flows = RFlows(*(inp[k].to(device) for k in ("fwd", "bwd", "fmask", "bmask")))
    tracks = [RTracks(xy.to(device), vis.to(device), s) for xy, vis, s in synthetic_track_arrays(frames, seed=seed)]
    opt = torch.optim.Adam(model.parameters(), lr=3e-5)  # model_wrapper_overfit.py:104-105, overfit.yaml:30
    state = {"step": START_STEP}

    def step():
        opt.zero_grad()
        gs = state["step"]
        out = model(batch, flows, gs)
        total = sum(l.forward(batch, flows, tracks, out, gs) for l in losses)
        total.backward()
        opt.step()
        state["step"] += 1
        return float(total.detach())
    return step


def reference_cpu(steps, warmup, budget_s=420.0):
    """`steps` timed iterations of the full C3 workload through the unmodified reference on the host
    cores (fixed thread policy: min(cores, 32) ATen threads -- ATen's elementwise kernels stop
    scaling well below 128 threads); the number of timed steps shrinks (>= 2) only if the first
    iteration shows that the run would not end within a few minutes."""
    cores = os.cpu_count() or 1
    threads = min(cores, 32)
    torch.set_num_threads(threads)
    step = reference_runner(torch.device("cpu"))
    t0 = time.perf_counter()
    first_loss = step()                       # untimed: first touch of 17 GB of autograd buffers
    t_first = time.perf_counter() - t0
    warm_done = 1
    while warm_done < warmup and (warm_done + 2) * t_first < 0.3 * budget_s:
        step()
        warm_done += 1
    k = max(2, min(steps, int((budget_s - warm_done * t_first) / max(t_first, 1e-3))))
    t0 = time.perf_counter()
    for _ in range(k):
        last = step()
    dt = (time.perf_counter() - t0) / k
    return {"value": 1.0 / dt, "unit": "it/s", "cores": cores, "threads": threads, "kind": "reference",
            "s_per_iteration": dt, "timed_steps": k, "warmup_steps": warm_done, "first_loss": first_loss,
            "last_loss": last,
            "sample": f"the full C3 workload (150 x 360 x 640, softmin + flow + tracking + Adam), {k} timed "
                      f"iterations after {warm_done} warm-up, unmodified reference modules (baseline/_ref) on "
                      f"{threads} ATen threads of {cores} host cores"}


# ------------------------------------------------------------------------------ CPU baseline (oracle port)
def cpu_baseline(sample_frames, steps, warmup, full=True):
    """The oracle (CPU restatement of the reference, oracle/flowmap_oracle.py: same op
    sequence on ATen, autograd, torch.optim.Adam) timed on the host cores on the first
    `sample_frames` frames of the workload; it/s scaled by frame pairs."""
    from oracle import flowmap_oracle as O
    inputs = synthetic_inputs(sample_frames, H_, W_, seed=0)
    cores = os.cpu_count() or 1
    f, h, w = sample_frames, H_, W_
    flows = O.Flows(inputs["fwd"], inputs["bwd"], inputs["fmask"], inputs["bmask"])
    tracks = [O.Tracks(xy, vis, s) for xy, vis, s in synthetic_track_arrays(f)] if full else None
    kw = dict(intrinsics="softmin", use_tracking=True) if full else dict(intrinsics="regressed")

    def make(nf):
        st = O.OverfitOracle(O.OverfitConfig(**kw), nf, h, w)
        with torch.no_grad():
            st.depth.copy_(inputs["depth"][:nf])
            st.weights.copy_(inputs["wparam"][:nf - 1])
        st.global_step = START_STEP
        return st

    # "all the host threads it can use": ATen's elementwise kernels stop scaling (and then
    # collapse) far below the core count of a 128-core host, so pick the fastest setting.
    best, best_t = None, None
    small = O.Flows(*(t[:, :2] for t in (inputs["fwd"], inputs["bwd"], inputs["fmask"], inputs["bmask"])))
    for nt in sorted({cores, min(cores, 64), min(cores, 32), min(cores, 16), min(cores, 8)}):
        torch.set_num_threads(nt)
        st = O.OverfitOracle(O.OverfitConfig(intrinsics="regressed"), 3, h, w)
        st.training_step(small)
        t0 = time.perf_counter()
        st.training_step(small)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = nt, dt
    torch.set_num_threads(best)

    def timed(kw_, use_tracks, n):
        st = O.OverfitOracle(O.OverfitConfig(**kw_), f, h, w)
        with torch.no_grad():
            st.depth.copy_(inputs["depth"][:f])
            st.weights.copy_(inputs["wparam"][:f - 1])
        st.global_step = START_STEP
        tr = tracks if use_tracks else None
        for _ in range(warmup):
            st.training_step(flows, tr)
        t0 = time.perf_counter()
        for _ in range(n):
            st.training_step(flows, tr)
        return (time.perf_counter() - t0) / n

    pairs = f - 1
    if not full:
        dt = timed(dict(intrinsics="regressed"), False, steps)
        t150 = dt * (F_ - 1) / pairs
        parts = {"s_per_sample_step": dt}
        how = f"time scales with frame pairs: t150 = t_sample * {F_ - 1}/{pairs}"
    else:
        # Three cost components with different scaling: per frame pair (flow path), per
        # iteration (the 60-candidate sweep on the first pair) and per (source, target) frame
        # pair of a track segment.  Time the sample with each switched on in turn, then
        # assemble the cost of the 150-frame workload.
        n_aux = max(1, min(steps, 2))
        t_flow = timed(dict(intrinsics="regressed"), False, n_aux)
        t_soft = timed(dict(intrinsics="softmin"), False, n_aux)
        t_full = timed(dict(intrinsics="softmin", use_tracking=True), True, steps)
        seg_pairs_sample = sum(xy.shape[1] ** 2 for xy, _, _ in synthetic_track_arrays(f))
        seg_pairs_full = sum(xy.shape[1] ** 2 for xy, _, _ in synthetic_track_arrays(F_))
        c_sweep = max(t_soft - t_flow, 0.0)
        # the sample's 3 short segments are too small to time inside a multi-second step: time
        # the tracking loss (forward + backward) on ONE full-size segment (41 frames x 1225)
        fs = 41
        seg = [O.Tracks(xy, vis, 0) for xy, vis, _ in synthetic_track_arrays(fs, interval=10 ** 6, radius=fs)]
        k = O.intrinsics_from_focal(torch.tensor(0.85), h, w).expand(1, fs, 3, 3)
        ext = torch.eye(4).expand(1, fs, 4, 4).clone()
        ext[0, :, 0, 3] = 0.01 * torch.arange(fs)
        ext.requires_grad_(True)
        with torch.no_grad():
            surf = O.unproject(O.pixel_grid(h, w), 0.1 + 0.05 * torch.rand(1, fs, h, w), k[:, :, None, None])
        surf.requires_grad_(True)  # marginal cost of the tracking loss given the shared surfaces

        def track_once():
            surf.grad = None
            O.tracking_loss(surf, ext, k, seg).backward()
        track_once()
        t0 = time.perf_counter()
        for _ in range(n_aux):
            track_once()
        c_track = (time.perf_counter() - t0) / n_aux / (fs * fs)
        t150 = t_flow * (F_ - 1) / pairs + c_sweep + c_track * seg_pairs_full
        parts = {"s_flow_path_sample": t_flow, "s_softmin_sweep": c_sweep,
                 "s_tracking_per_frame_pair": c_track, "s_full_sample_step": t_full,
                 "track_frame_pairs_sample": seg_pairs_sample, "track_frame_pairs_150": seg_pairs_full}
        how = (f"t150 = t_flow_path * {F_ - 1}/{pairs} + t_sweep + t_track_per_frame_pair * "
               f"{seg_pairs_full} (tracking timed on one 41-frame x 1225-track segment)")
    return {"value": 1.0 / t150, "unit": "it/s", "cores": cores, "kind": "port", "threads": best,
            "frame_pairs_per_s": (F_ - 1) / t150, "estimated_s_per_iteration_150_frames": t150,
            "sample": f"first {f} of {F_} frames ({pairs} pairs, {len(tracks) if tracks else 0} track "
                      f"segments) at {h}x{w}, {steps} timed steps after {warmup} warm-up; {how}",
            **parts}


# ------------------------------------------------------------------------------ ncu evidence
NCU_SUMMARY = ROOT / "profiles" / "r2_path_ncu_summary.txt"  # tools/ncu_summary.py output, committed


def ncu_traffic_from_profiles(path=NCU_SUMMARY):
    """{op: dram bytes per launch} for the three pixel kernels from the committed ncu summary."""
    names = {"k_moments_dense": "procrustes_fwd(k_moments)", "k_flow_lean": "flow_loss_fwd_bwd(k_flow_lean)",
             "k_distribute_dense": "procrustes_bwd(k_distribute)"}
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    out, cur = {}, None
    if not Path(path).exists():
        return {}, None
    for line in Path(path).read_text().splitlines():
        if line.startswith("====="):
            cur = next((v for k, v in names.items() if f"::{k}<" in line or f"::{k}(" in line), None)
        elif cur and ("dram__bytes_read.sum " in line or "dram__bytes_write.sum " in line):
            parts = line.split()
            out[cur] = out.get(cur, 0.0) + float(parts[1]) * unit.get(parts[2], 1.0)
    return out, str(Path(path).relative_to(ROOT))


# ------------------------------------------------------------------------------ pair sharding
def device_shard_inputs(f, h, w, pair_lo, pair_hi, dev):
    """The frames [pair_lo, pair_hi] / pairs [pair_lo, pair_hi) of one synthetic video, generated on
    the device with per-frame / per-pair seeds: every rank builds exactly its shard of the SAME
    video whatever the world size (same distributions as synthetic_inputs)."""
    def gen(seed):
        return torch.Generator(device=dev).manual_seed(seed)
    nf = pair_hi - pair_lo + 1
    depth = torch.empty(nf, h, w, device=dev)
    for i in range(nf):
        depth[i] = 0.1 + 0.05 * torch.rand(h, w, device=dev, generator=gen(10_000 + pair_lo + i))
    npair = pair_hi - pair_lo
    wparam = torch.empty(npair, h, w, device=dev)
    fwd, bwd = torch.empty(1, npair, h, w, 2, device=dev), torch.empty(1, npair, h, w, 2, device=dev)
    fm, bm = torch.empty(1, npair, h, w, device=dev), torch.empty(1, npair, h, w, device=dev)
    for i in range(npair):
        g = gen(20_000 + pair_lo + i)
        wparam[i] = 0.01 * torch.randn(h, w, device=dev, generator=g)
        fwd[0, i] = 0.01 * torch.randn(h, w, 2, device=dev, generator=g)
        bwd[0, i] = 0.01 * torch.randn(h, w, 2, device=dev, generator=g)
        fm[0, i] = torch.rand(h, w, device=dev, generator=g)
        bm[0, i] = torch.rand(h, w, device=dev, generator=g)
    return depth, wparam, (fwd, bwd, fm, bm)


def sharded_record(f, h, w, full, rank, world, dev, steps, barrier, max_over_ranks):
    """Strong scaling of ONE f x h x w video over the ranks of this run: ms/step with its pairs
    split over `world` ranks, the same video on one rank (rank 0) alongside, bytes sent per rank per
    step and the device time inside the exchange (CUDA events around every collective / the two
    halves of StepReducer on the step's stream, eager steps; includes waiting for the slowest
    neighbour; in the flow-only step Adam on the interior frames runs between the two halves)."""
    from flowmap_b200 import parallel
    from flowmap_b200.overfit import OverfitCfg, ShardedFusedOverfitter
    from flowmap_b200.types import Batch, Flows, Tracks

    def build(plan, group=None):
        a, b = plan.pair_range
        depth, wparam, fl = device_shard_inputs(f, h, w, a, b, dev)
        nf = b - a + 1
        batch = Batch(torch.zeros(1, 1, 1, 1, 1, device=dev).expand(1, nf, 3, h, w),
                      torch.arange(nf, device=dev)[None], ["synthetic"], ["synthetic"])
        cfg = OverfitCfg(intrinsics="softmin", use_tracking=True) if full else OverfitCfg()
        tracks = [Tracks(xy, vis, s) for xy, vis, s in synthetic_track_arrays(f, seed=0)] if full else None
        o = ShardedFusedOverfitter(cfg, batch, Flows(*fl), plan, tracks=tracks, device=dev, group=group)
        o.use_cuda_graph = os.environ.get("FM_BENCH_NO_GRAPH") != "1"
        with torch.no_grad():
            o.model.backbone.depth.copy_(depth)
            o.model.backbone.weights.copy_(wparam)
        o.global_step = START_STEP
        return o

    def timed(o, n):
        for _ in range(3):
            o.training_step()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(n):
            o.training_step()
        e1.record()
        barrier()
        return e0.elapsed_time(e1) / n

    plan = parallel.make_plan(f - 1, rank, world)
    o = build(plan)
    ms_n = max_over_ranks(timed(o, steps))
    # time inside the exchange: CUDA events around every collective of a few extra steps (the
    # blocking collectives make the step's stream wait for the NCCL stream, so the events bracket
    # them; StepReducer.reduce is bracketed as a whole: grouped send/recv + all-reduce + the two adds)
    import torch.distributed as dist
    spans, depth = [], {"n": 0}

    def wrap(fn):
        def inner(*a, **k):
            if depth["n"] > 0:  # a collective inside an already bracketed exchange
                return fn(*a, **k)
            depth["n"] += 1
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            try:
                return fn(*a, **k)
            finally:
                e1.record()
                spans.append((e0, e1))
                depth["n"] -= 1
        return inner
    real = (o.reducer.reduce, o.reducer.start, o.reducer.finish, dist.all_reduce, dist.broadcast)
    (o.reducer.reduce, o.reducer.start, o.reducer.finish, dist.all_reduce, dist.broadcast) = (wrap(f) for f in real)
    n_probe = 5
    graph_was = o.use_cuda_graph
    o.use_cuda_graph = False  # the probes are host-side wrappers: run these steps eagerly
    try:
        barrier()
        for _ in range(n_probe):
            o.training_step()
        torch.cuda.synchronize()
    finally:
        o.reducer.reduce, o.reducer.start, o.reducer.finish, dist.all_reduce, dist.broadcast = real
        o.use_cuda_graph = graph_was
    comm_ms = max_over_ranks(sum(a.elapsed_time(b) for a, b in spans) / n_probe)
    sent = o.reducer.bytes_per_step()
    o_graph = bool(o._graphs)
    del o
    torch.cuda.empty_cache()
    ms_1 = None
    if world == 1:
        ms_1 = ms_n
    else:  # the same video unsharded, on rank 0 alone (the others wait at the barrier)
        g0 = torch.distributed.new_group([0])  # collective: every rank creates the one-rank group
        if rank == 0:
            solo = build(parallel.ShardPlan(0, 1, (0, f - 1), f - 1), group=g0)
            for _ in range(3):
                solo.training_step()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(steps):
                solo.training_step()
            e1.record()
            torch.cuda.synchronize()
            ms_1 = e0.elapsed_time(e1) / steps
            del solo
        t = torch.tensor([ms_1 if ms_1 is not None else 0.0], device=dev, dtype=torch.float64)
        torch.distributed.broadcast(t, src=0)
        ms_1 = float(t)
    return {"frames": f, "height": h, "width": w, "pairs": f - 1, "n_gpus": world,
            "what": ("full loop (softmin sweep on rank 0, tracking sharded by source frame)" if full
                     else "flow loss only, regressed focal (BASELINE configs[3])"),
            "ms_per_step": round(ms_n, 4), "ms_per_step_one_gpu": round(ms_1, 4),
            "speedup": round(ms_1 / ms_n, 3), "strong_scaling_efficiency": round(ms_1 / ms_n / world, 4),
            "it_per_s": round(1000.0 / ms_n, 2), "bytes_sent_per_rank_per_step": int(sent),
            "ms_in_exchange_per_step": round(comm_ms, 4), "cuda_graph": bool(o_graph),
            "exchange": "one 2-float all-reduce + one boundary depth-gradient frame swapped with each neighbour"
                        + (" + pose gather, tracking-sum all-reduce (F x 10 doubles), focal broadcast" if full else "")}


# ------------------------------------------------------------------------------ GPU arm
def run_gpu(args):
    from flowmap_b200 import ops, parallel
    from flowmap_b200._lib import lib
    from flowmap_b200.overfit import FusedOverfitter, OverfitCfg, ShardedFusedOverfitter
    from flowmap_b200.types import Batch, Flows, Tracks

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (flowmap_b200 has no CPU path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    pairs_mode = args.mode in ("pairs", "pairs-full")
    pairs_full = args.mode == "pairs-full"

    # the step clock draws the seed of its softmin point sample from torch's generator
    torch.manual_seed(rank)
    inputs = synthetic_inputs(F_, H_, W_, seed=rank)
    batch = Batch(torch.zeros(1, 1, 1, 1, 1, device=dev).expand(1, F_, 3, H_, W_),
                  torch.arange(F_, device=dev)[None], ["synthetic"], ["synthetic"])
    flows_host = Flows(inputs["fwd"].pin_memory(), inputs["bwd"].pin_memory(),
                       inputs["fmask"].pin_memory(), inputs["bmask"].pin_memory())

    def device_flows():
        return Flows(*(t.to(dev, non_blocking=True) for t in
                       (flows_host.forward, flows_host.backward, flows_host.forward_mask,
                        flows_host.backward_mask)))

    def init_params(o):
        with torch.no_grad():
            o.model.backbone.depth.copy_(inputs["depth"])
            o.model.backbone.weights.copy_(inputs["wparam"])
        o.global_step = START_STEP
        return o

    flows_dev = device_flows()
    if pairs_mode:
        plan = parallel.ShardPlan(rank, world, (rank * (F_ - 1), (rank + 1) * (F_ - 1)), world * (F_ - 1))
        if pairs_full:  # one long video, full loop: global track segments, sweep on rank 0
            tracks = [Tracks(xy, vis, s) for xy, vis, s in synthetic_track_arrays(world * (F_ - 1) + 1, seed=0)]
            o = init_params(ShardedFusedOverfitter(OverfitCfg(intrinsics="softmin", use_tracking=True), batch,
                                                   flows_dev, plan, tracks=tracks, device=dev))
        else:
            o = init_params(ShardedFusedOverfitter(OverfitCfg(), batch, flows_dev, plan, device=dev))
        o.sync_boundary_depth()
    else:
        tracks = [Tracks(xy, vis, s) for xy, vis, s in synthetic_track_arrays(F_, seed=rank)]
        o = init_params(FusedOverfitter(OverfitCfg(intrinsics="softmin", use_tracking=True), batch,
                                        flows_dev, tracks, device=dev))
        o.use_cuda_graph = os.environ.get("FM_BENCH_NO_GRAPH") != "1"  # the step replayed as one CUDA graph

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        t = torch.tensor([v], device=dev, dtype=torch.float64)
        if world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return float(t)

    def time_steps(fn, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        t0 = time.time()
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        barrier()
        clocks.window(t0, time.time())
        return max_over_ranks(e0.elapsed_time(e1) / steps), out

    # ---- parity gate: the first step of THIS workload (seed 0) against the value the unmodified
    # reference produced for it (tests/golden/big_c3.npz, generated by tests/golden/make_golden_big.py
    # with the same softmin point indices); a fast step that computes something else is worthless
    loss_check = None
    fixture = ROOT / "tests" / "golden" / "big_c3.npz"
    if not pairs_mode and rank == 0 and fixture.exists():
        import numpy as np
        with np.load(fixture) as z:
            ref_loss, ref_idx = float(z["loss"][0]), torch.as_tensor(z["softmin_indices"])
        o.injected_indices = ref_idx.to(dev)
        got = float(o.training_step(update=False)[0])
        o.injected_indices = None
        rel_err = abs(got - ref_loss) / abs(ref_loss)
        loss_check = {"step0_loss": got, "reference_step0_loss": ref_loss, "rel_err": rel_err, "tolerance": 1e-4,
                      "source": "tests/golden/big_c3.npz (unmodified reference, float32, CPU)"}
        if not rel_err <= 1e-4:
            raise SystemExit(f"bench.py: step-0 loss {got} differs from the reference's {ref_loss} (rel {rel_err:.2e})")

    # ---- device-resident timing (value)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    l0 = lib().fm_launch_count()
    o.training_step()  # the first warm-up step runs eagerly: its launches are the step's kernel list
    launches_per_step = lib().fm_launch_count() - l0
    for _ in range(max(args.warmup, 4) - 1):  # (the graph is captured on the third step)
        o.training_step()
    l0 = lib().fm_launch_count()
    ms, last = time_steps(o.training_step, args.steps)
    launches = lib().fm_launch_count() - l0
    if args.dump_outputs and rank == 0:  # before the legs below run more steps on `o`
        dump_outputs(args.dump_outputs, o, last)
    graph_replay = bool(getattr(o, "_graphs", None))
    if graph_replay:  # replayed graph nodes are not host launches: count the kernels they contain
        launches = launches_per_step * args.steps
    final_loss = float(last[0])

    # ---- end-to-end: the step's Flows arrive in pinned host memory every step (the
    # pretrain-style use of the same API), the loss is read back to the host every step.
    h2d = sum(x.numel() * 4 for x in (flows_host.forward, flows_host.backward,
                                      flows_host.forward_mask, flows_host.backward_mask))

    # Double-buffered, as a prefetching loader would do it: while step k computes on one device
    # buffer, the copy engine uploads step k+1's Flows into the other (every step still moves its
    # 824 MB inside the timed region; the copy just overlaps the previous step's kernels).
    fields = ("forward", "backward", "forward_mask", "backward_mask")
    bufs = [o.flows, Flows(*(torch.empty_like(getattr(o.flows, n)) for n in fields))]
    copy_stream = torch.cuda.Stream()
    main_stream = torch.cuda.current_stream()
    ready = [torch.cuda.Event(), torch.cuda.Event()]  # upload into buffer i finished
    free = [torch.cuda.Event(), torch.cuda.Event()]   # kernels reading buffer i finished
    for ev in free:
        ev.record(main_stream)
    turn = {"i": 0}

    def upload(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(free[i])
            for n in fields:
                getattr(bufs[i], n).copy_(getattr(flows_host, n), non_blocking=True)
            ready[i].record(copy_stream)

    upload(0)

    def e2e_step():
        i = turn["i"]
        turn["i"] = i ^ 1
        main_stream.wait_event(ready[i])
        upload(i ^ 1)                 # next step's inputs travel while this step computes
        o.set_flows(bufs[i])          # masks are "new": the normaliser is recomputed (all-reduced if sharded)
        loss = o.training_step()[0]
        free[i].record(main_stream)
        return float(loss)            # D2H read of the step's loss

    for _ in range(2):
        e2e_step()
    e2e_ms, _ = time_steps(e2e_step, max(3, min(args.steps, 10)))

    # ---- flow-loss-only variant of the same step (regressed focal): the path the roofline
    # accounting below describes; and the same on spatially smooth flows (real optical flow is
    # piecewise smooth; the iid flows above are the worst case for the bilinear gather/scatter)
    flow_only_ms = smooth_ms = sparse_ms = dropin_ms = None
    if not pairs_mode:
        o2 = init_params(FusedOverfitter(OverfitCfg(), batch, flows_dev, device=dev))
        for _ in range(3):
            o2.training_step()
        flow_only_ms, _ = time_steps(o2.training_step, min(args.steps, 30))
        g = torch.Generator(device=dev).manual_seed(rank)
        for t in (o2.flows.forward, o2.flows.backward):
            lo = 0.01 * torch.randn(F_ - 1, 2, H_ // 16 + 1, W_ // 16 + 1, device=dev, generator=g)
            up = torch.nn.functional.interpolate(lo, size=(H_, W_), mode="bilinear", align_corners=True)
            t.copy_(up.permute(0, 2, 3, 1)[None])
        for _ in range(3):
            o2.training_step()
        smooth_ms, _ = time_steps(o2.training_step, min(args.steps, 30))
        del o2
        flows_dev.forward.copy_(flows_host.forward, non_blocking=True)
        flows_dev.backward.copy_(flows_host.backward, non_blocking=True)
        # the reference's DEFAULT pose solve uses 1000 evenly spaced points per pair
        # (config/model/extrinsics/procrustes.yaml:3-4) instead of all pixels
        o3 = init_params(FusedOverfitter(OverfitCfg(procrustes_points=1000), batch, flows_dev, device=dev))
        for _ in range(3):
            o3.training_step()
        sparse_ms, _ = time_steps(o3.training_step, min(args.steps, 30))
        del o3
        # the SAME full workload through the per-module drop-in surface (Model.forward, LossFlow /
        # LossTracking.forward as autograd Functions, Adam on the kernel): what install() gives the
        # reference's own training loop, one C-ABI call per op instead of one per step
        from flowmap_b200.overfit import Overfitter
        o4 = init_params(Overfitter(OverfitCfg(intrinsics="softmin", use_tracking=True), batch, flows_dev,
                                    tracks, device=dev))
        for _ in range(3):
            o4.training_step()
        dropin_ms, _ = time_steps(o4.training_step, min(args.steps, 20))
        del o4
        flows_dev.forward.copy_(flows_host.forward, non_blocking=True)   # o.flows shares these buffers
        flows_dev.backward.copy_(flows_host.backward, non_blocking=True)

    # ---- pair-sharded strong scaling, measured in the same run (SURVEY 8(e), BASELINE configs[3]):
    # ONE video, its frame pairs split over the N ranks; per step one 2-float all-reduce and one
    # boundary depth-gradient frame swapped with each neighbour (NCCL over NVLink).
    pair_sharded = None
    if not pairs_mode and os.environ.get("FM_BENCH_SKIP_SHARDED") != "1":
        pair_sharded = {}
        for name, (pf, ph, pw, full) in {"config4_flow_only": (150, 720, 1280, False),
                                         "config3_full_loop": (F_, H_, W_, True)}.items():
            if name == "config3_full_loop" and world == 1:
                continue  # at N = 1 this is the headline `value` itself
            try:
                pair_sharded[name] = sharded_record(pf, ph, pw, full, rank, world, dev, max(5, min(args.steps, 30)),
                                                    barrier, max_over_ranks)
            except Exception as exc:  # noqa: BLE001 -- keep the bench line
                pair_sharded[name] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
            torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            torch.distributed.barrier()  # rank 0 still runs its per-op timing / CPU baseline
            torch.distributed.destroy_process_group()
        return

    # ---- per-op timing for the roofline (rank 0; ops called through the C ABI, CUDA events on
    # the launching stream)
    with torch.no_grad():
        depths = o.model.backbone.depth.detach()[None].contiguous()
        weights = torch.sigmoid(100.0 * o.model.backbone.weights.detach())[None].contiguous()
        s_ = (H_ * W_) ** 0.5
        k4 = torch.tensor([0.85 * s_ / W_, 0.85 * s_ / H_, 0.5, 0.5], device=dev).expand(1, F_, 4).contiguous()
        msum = ops.mask_sum(o.flows.forward_mask, o.flows.backward_mask)
        ws = ops.workspace(1, F_, H_, W_, dev)
        rt = torch.empty(1, F_ - 1, 3, 4, device=dev)
        g_depth, g_w = torch.empty_like(depths), torch.empty_like(weights)
        g_k4, g_rt = torch.empty_like(k4), torch.empty_like(rt)
        lossb = torch.empty((), device=dev)
        P = lambda x: x.data_ptr()  # noqa: E731
        st = torch.cuda.current_stream().cuda_stream
        L = lib()
        fl = o.flows

        def op_fwd():
            L.fm_procrustes_fwd(P(depths), P(k4), P(fl.backward), P(weights), None, 0, P(rt), P(ws),
                                1, F_, H_, W_, st)

        def op_flow():
            L.fm_flow_loss_fwd_bwd(P(depths), P(k4), P(rt), P(fl.forward), P(fl.backward),
                                   P(fl.forward_mask), P(fl.backward_mask), P(msum), 0, 0.01, 1000.0,
                                   1, P(lossb), P(g_depth), P(g_rt), P(g_k4), P(ws), 1, F_, H_, W_, st)

        def op_bwd():
            L.fm_procrustes_bwd(P(depths), P(k4), P(fl.backward), P(weights), None, 0, None, 1, None,
                                P(g_depth), P(g_w), P(g_k4), P(ws), 1, F_, H_, W_, st)

        def timed(fn, n=10):
            for _ in range(3):
                op_fwd(); op_flow(); fn()
            torch.cuda.synchronize()
            tot = 0.0
            for _ in range(n):
                if fn is op_bwd:
                    op_flow()  # re-create the direct gradient that op_bwd accumulates into
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); fn(); b.record()
                torch.cuda.synchronize()
                tot += a.elapsed_time(b)
            return tot / n
        t_fwd, t_flow, t_bwd = timed(op_fwd), timed(op_flow), timed(op_bwd)
    clk = clocks.stop()

    peaks_path = ROOT / "MEASURED_PEAKS.json"
    if peaks_path.exists():
        peak, peak_src = json.loads(peaks_path.read_text())["hbm_gbs"], "measured (MEASURED_PEAKS.json)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    n, p_ = H_ * W_, F_ - 1
    ops_bytes = {  # algorithmic bytes per launch: inputs read once, outputs written once
        "procrustes_fwd(k_moments)": n * (4 * F_ + (8 + 4) * p_),
        "flow_loss_fwd_bwd(k_flow_lean)": n * (4 * F_ + (8 + 8 + 4 + 4) * p_ + 4 * F_),
        "procrustes_bwd(k_distribute)": n * (4 * F_ + (8 + 4) * p_ + 4 * p_ + 8 * F_),
    }
    times = {"procrustes_fwd(k_moments)": t_fwd, "flow_loss_fwd_bwd(k_flow_lean)": t_flow,
             "procrustes_bwd(k_distribute)": t_bwd}
    dom = max(times, key=times.get)
    path_ms = t_fwd + t_flow + t_bwd
    path_gbs = algorithmic_bytes(F_, H_, W_) / (path_ms * 1e-3) / 1e9
    dom_gbs = ops_bytes[dom] / (times[dom] * 1e-3) / 1e9
    # DRAM bytes per launch: parsed from the committed `ncu --set full` summary of these kernels at
    # this shape (dram__bytes_read.sum + dram__bytes_write.sum); None if the file is missing
    ncu_traffic, traffic_file = ncu_traffic_from_profiles()
    roofline = {"bound": "hbm", "kernel": dom, "achieved": round(dom_gbs, 1), "peak": peak,
                "unit": "GB/s", "frac": round(dom_gbs / peak, 4), "traffic": ncu_traffic.get(dom),
                "algorithmic_bytes": ops_bytes[dom],
                "traffic_source": f"ncu --set full capture of this kernel at this shape ({traffic_file})",
                "path_traffic": (sum(ncu_traffic.values()) if len(ncu_traffic) == 3 else None),
                "peak_source": peak_src,
                "path": {"what": "unproject->Procrustes->reproject->loss+grad (3 ops, summed)",
                         "algorithmic_bytes": algorithmic_bytes(F_, H_, W_),
                         "ms": round(path_ms, 4), "achieved": round(path_gbs, 1),
                         "frac": round(path_gbs / peak, 4)},
                "ops_ms": {k: round(v, 4) for k, v in times.items()},
                "note": "k_distribute is bound by L2 RED (atomic add) throughput, k_flow_lean by exposed "
                        "load latency at 2 CTAs/SM (128 registers), k_moments by L1 gather wavefronts "
                        "(profiles/README.md); HBM is the denominator the task names"}

    # ---- informative: the unmodified reference in its own execution mode, CUDA eager on this same
    # B200 (flowmap/overfit.py:50,96 hard-code cuda:0) -- what a FlowMap user runs today
    ref_cuda = None
    if world == 1 and not pairs_mode and reference_available() and os.environ.get("FM_BENCH_SKIP_CPU") != "1":
        try:
            del o
            torch.cuda.empty_cache()
            rstep = reference_runner(dev)
            rstep(); rstep()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            n_ref = 5
            for _ in range(n_ref):
                rl = rstep()
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) / n_ref
            ref_cuda = {"ms_per_step": round(dt * 1e3, 2), "it_per_s": round(1.0 / dt, 3), "steps": n_ref,
                        "last_loss": rl, "peak_mem_gb": round(torch.cuda.max_memory_allocated() / 2 ** 30, 1),
                        "what": "unmodified reference modules (baseline/_ref) in PyTorch CUDA eager on this GPU, same "
                                "workload, wall clock with a synchronize on both sides (loss read back every step)"}
            del rstep
            torch.cuda.empty_cache()
        except Exception as exc:  # noqa: BLE001 -- the informative leg must not sink the bench line
            ref_cuda = {"error": f"{type(exc).__name__}: {exc}"[:300]}

    if os.environ.get("FM_BENCH_SKIP_CPU") == "1":  # profiling runs (ncu) only
        cpu = {"value": None, "unit": "it/s", "cores": os.cpu_count(), "kind": "port",
               "sample": "skipped (FM_BENCH_SKIP_CPU=1)"}
    elif world > 1:  # the CPU baseline is a property of the host, timed in the N=1 run
        cpu = {"value": None, "unit": "it/s", "cores": os.cpu_count(), "kind": "port",
               "sample": "timed on rank 0 at N=1 only (see the --gpus 1 line)"}
    else:
        cpu = cpu_baseline(sample_frames=12, steps=2, warmup=1, full=not pairs_mode or pairs_full)

    its = world * 1000.0 / ms
    out = {
        "metric": METRIC, "value": round(its, 3), "unit": "it/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 4),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "frame_pairs_per_s": round(its * (F_ - 1), 1),
        "config": {"workload": WORKLOAD if (not pairs_mode or pairs_full) else
                   WORKLOAD.replace("softmin intrinsics (60 candidates x 8192 points), flow + tracking loss",
                                    "regressed focal, flow loss only"),
                   "frames": F_, "height": H_, "width": W_,
                   "parallelism": ("%d independent scenes, one per GPU (BASELINE config 5), no "
                                   "collective" % world) if not pairs_mode else
                                  ("%d x %d pairs of one video; per step a 2-float all-reduce and one boundary "
                                   "frame swapped with each neighbour (%d bytes sent per rank)"
                                   % (world, F_ - 1, o.reducer.bytes_per_step())) +
                                  (" + pose gather, tracking-sum all-reduce (F x 10 doubles), focal broadcast"
                                   if pairs_full else ""),
                   "l2": "inputs (1.1 GB) exceed the 126 MB L2, no flush needed",
                   "mask_sum": "loop-invariant flow-loss denominator hoisted out of the loop "
                               "(recomputed every step in the e2e leg, where the masks are re-uploaded)"},
        "e2e": {"value": round(world * 1000.0 / e2e_ms, 3), "unit": "it/s",
                "ms_per_step": round(e2e_ms, 3), "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "what": "Flows (flow fwd/bwd + masks) copied from pinned host memory every step "
                        "(double-buffered: step k+1 uploads while step k computes), loss read back "
                        "every step"},
        "gpu_launches": int(launches), "launches_per_step": int(launches_per_step),
        "cuda_graph": graph_replay, "final_loss": final_loss, "loss_check": loss_check,
        "flow_only": None if flow_only_ms is None else
        {"ms_per_step": round(flow_only_ms, 4), "it_per_s": round(world * 1000.0 / flow_only_ms, 2),
         "what": "same step without tracking loss / softmin sweep (regressed focal)",
         "ms_per_step_smooth_flows": None if smooth_ms is None else round(smooth_ms, 4),
         "ms_per_step_1000_point_procrustes": None if sparse_ms is None else round(sparse_ms, 4),
         "smooth_flows": "N(0, 0.01^2) flow on a 16x coarser grid, bilinearly upsampled"},
        "dropin_autograd": None if dropin_ms is None else
        {"ms_per_step": round(dropin_ms, 4), "it_per_s": round(world * 1000.0 / dropin_ms, 2),
         "what": "same full workload through Model.forward + LossFlow/LossTracking autograd Functions + "
                 "kernel Adam (the install() drop-in surface) instead of the one-call fused step"},
        "pair_sharded": pair_sharded,
        "reference_cuda_eager": ref_cuda,
        "clocks": clk, "roofline": roofline, "cpu_baseline": cpu,
    }
    print(json.dumps(out))
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


# ------------------------------------------------------------------------------ reference arm
def run_reference(args):
    """The reference's own CPU implementation of the path: the UNMODIFIED reference modules staged
    under baseline/_ref (baseline/install_ref.py) on the full C3 workload; if they are missing
    (baseline/install_ref.py was not run) the oracle port on a bounded sample, labelled as such."""
    if int(os.environ.get("RANK", 0)) != 0:
        return
    if reference_available() and args.mode == "scenes":
        cpu = reference_cpu(max(2, args.steps), max(1, args.warmup))
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": round(cpu["value"], 6), "unit": "it/s",
            "n_gpus": int(os.environ.get("WORLD_SIZE", 1)), "steps": cpu["timed_steps"], "warmup": cpu["warmup_steps"],
            "requested_steps": args.steps, "ms_per_step": round(1000.0 * cpu["s_per_iteration"], 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "frames": F_, "height": H_, "width": W_},
            "cpu_baseline": cpu,
            "e2e": {"value": round(cpu["value"], 6), "unit": "it/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0},
            "gpu_launches": 0}))
        return
    # exactly K timed steps; the sample shrinks with K so that the run stays within minutes
    frames = max(3, min(12, 60 // max(1, args.steps) + 2))
    cpu = cpu_baseline(sample_frames=frames, steps=max(1, args.steps),
                       warmup=max(1, min(args.warmup, 2)), full=args.mode != "pairs")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": round(cpu["value"], 6), "unit": "it/s",
        "n_gpus": int(os.environ.get("WORLD_SIZE", 1)), "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(1000.0 / cpu["value"], 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": WORKLOAD},
        "cpu_baseline": cpu,
        "e2e": {"value": round(cpu["value"], 6), "unit": "it/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="scenes", choices=["scenes", "pairs", "pairs-full"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        args.warmup = max(args.warmup, 3)
        run_gpu(args)


if __name__ == "__main__":
    main()
