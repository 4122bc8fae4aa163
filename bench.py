#!/usr/bin/env python
"""bench.py -- rollout cost+gradient throughput, (seed x waypoint) evals/s.

    python bench.py --gpus N --steps K --warmup W [--workload NAME] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the fused rollout kernel over one batch of synthetic joint configurations
(= what one optimizer iteration's cost+gradient evaluation does, gradient_opt_core.py:445-480).
Default workload = BASELINE.json configs[1]: Franka IK, 512 targets x 32 seeds (16,384 evals/step),
primitive-cuboid world, H = 1.  N > 1: the seed batch is sharded (weak scaling: 16,384 evals per GPU),
no data-path collective; one NCCL all_gather of per-seed costs after the timed region (not timed:
it happens once per solve, not per iteration).

Prints ONE JSON line (rank 0).  `value` = device-resident throughput (CUDA events per step on the
launching stream, L2 flushed between steps, max over ranks; `value_warm_l2` = the same loop without the
flush); `e2e` = same metric through the public API with pinned-host inputs and host read-back inside the
timed region (one CUDA graph per step: H2D, kernel, D2H; no flush -- the inputs arrive by H2D every step);
`roofline` = algorithmic bytes per eval (BASELINE.md section 4) x evals / kernel time vs the measured HBM
peak; `cpu_baseline` = the numpy oracle (a port of the reference arithmetic; the reference has no CPU
path) on a bounded sample.  `sharded` = BASELINE configs 4 and 5 STRONG-scaled over the N ranks (total rows
fixed, rows / N per rank): rollout-only and a complete seed-sharded L-BFGS solve with the end-of-solve
all_gather inside the timed region.  `baseline_configs` (last key, compact) = configs 2-5 on one line.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "rollout_cost_grad_evals_per_sec"
UNIT = "evals/s"


# ------------------------------------------------------------------------------------------------
# workloads (BASELINE.md section 3)
# ------------------------------------------------------------------------------------------------
def make_workload(name: str, seed_offset: int = 0):
    """`<workload>_dynamics` / `<workload>_dynamics_host`: the same rows with the dynamics-aware STATE cost (SURVEY.md 8f rank 3),
    evaluated inside the trajectory kernel or by the three extra launches of the host composition (synthetic inertial parameters)."""
    mode = None
    for suffix, m in (("_dynamics_host", "host"), ("_dynamics", "fused")):
        if name.endswith(suffix):
            name, mode = name[:-len(suffix)], m
            break
    wl = _make_workload(name, seed_offset)
    wl["dynamics"] = mode
    if mode is not None and "mpc" in name:
        # the effort channel has zero weight in lbfgs_mpc.yml; the dynamics-aware variants keep the trajopt weights
        # (effort bound 100, energy 10000) they were introduced with
        from curobo_b200.rollout import RolloutConfig
        wl["cfg"] = RolloutConfig.trajopt()
        wl.pop("cs_target", None)
    return wl


def _make_workload(name: str, seed_offset: int = 0):
    """Returns dict(robot, cfg, B, H, q [B,H,D] np, goal (pos, quat, idx) or None, cuboid world, voxel spec, bytes_per_eval)."""
    from curobo_b200.robot_model import load_robot
    from curobo_b200.rollout import RolloutConfig
    from curobo_b200.world import make_benchmark_cuboid_world
    from helpers import random_q
    from oracle import rollout_oracle as O
    if name == "franka_ik_512x32_cuboid":
        rm = load_robot("franka")
        B, H = 512 * 32, 1
        q = random_q(rm, B, seed=100 + seed_offset)[:, None, :]
        _, _, gp, gq = O.fk_forward(rm, random_q(rm, 512, seed=7))
        goal = (gp[:, :, None, :].copy(), gq[:, :, None, :].copy(), (np.arange(B) // 32).astype(np.int32))
        D, S, L = rm.num_dof, rm.num_spheres, rm.num_tool_frames
        bpe = 4 * D + 4 * D + 4 * (S + 1 + 2 * L + D)                      # 356 B, cuboid world: no obstacle bytes
        return dict(robot=rm, cfg=RolloutConfig.ik(), B=B, H=H, q=q, goal=goal, cuboid=make_benchmark_cuboid_world(),
                    voxel=None, bytes_per_eval=bpe)
    if name in ("g1_29_8192_esdf", "g1_43_8192_esdf", "franka_16384_esdf"):
        rname = {"g1_29_8192_esdf": "g1_29", "g1_43_8192_esdf": "g1_43", "franka_16384_esdf": "franka"}[name]
        rm = load_robot(rname)
        B, H = (16384 if rname == "franka" else 8192), 1
        from helpers import humanoid_q
        q = (humanoid_q(rm, B, seed=200 + seed_offset) if rname != "franka" else random_q(rm, B, seed=200 + seed_offset))[:, None, :]
        D, S, L = rm.num_dof, rm.num_spheres, rm.num_tool_frames
        bpe = 4 * D + 4 * D + 4 * (S + 1 + 2 * L + D) + 16 * S             # + 8 fp16 corners per sphere
        cfg = RolloutConfig(self_weight=5000.0, scene_weight=5000.0, scene_activation=0.02, cspace_type="position",
                            cspace_weight=(5000.0, 0, 0, 0, 0), cspace_activation=(0.01, 0, 0, 0, 0))
        return dict(robot=rm, cfg=cfg, B=B, H=H, q=q, goal=None, cuboid=None, voxel=dict(n=256, voxel=0.01, boxes=12, seed=0),
                    bytes_per_eval=bpe)
    if name in ("franka_mpc_1024x30_esdf_swept", "franka_trajopt_32x32_esdf_swept"):
        from helpers import random_walk_q
        rm = load_robot("franka")
        B, H = (1024, 30) if "mpc" in name else (32, 32)
        q = random_walk_q(rm, B, H, seed=300 + seed_offset)
        vel = (np.gradient(q, axis=1) / 0.05).astype(np.float32)
        acc = (np.gradient(vel, axis=1) / 0.05).astype(np.float32)
        jerk = (np.gradient(acc, axis=1) / 0.05).astype(np.float32)
        _, _, gp, gq = O.fk_forward(rm, random_q(rm, B, seed=9))
        goal = (gp[:, :, None, :].copy(), gq[:, :, None, :].copy(), np.arange(B, dtype=np.int32))
        D, S, L = rm.num_dof, rm.num_spheres, rm.num_tool_frames
        bpe = 4 * D + 4 * D + 4 * (S + 1 + 2 * L + D) + 16 * S * 7 + 3 * 4 * D * 2   # swept worst case n_s = 7; v/a/j in + grads out
        # config 4 (MPC) runs the shipped MPC weights (lbfgs_mpc.yml: c-space target term at 1000, x0.05 on non-terminal
        # waypoints); config 3 (trajopt) the shipped B-spline trajopt weights
        mpc = "mpc" in name
        wl = dict(robot=rm, cfg=RolloutConfig.mpc() if mpc else RolloutConfig.trajopt(), B=B, H=H, q=q, goal=goal, cuboid=None,
                  voxel=dict(n=256, voxel=0.01, boxes=12, seed=0), bytes_per_eval=bpe,
                  extra=dict(vel=vel, acc=acc, jerk=jerk, dt=np.full(B, 0.05, np.float32)))
        if mpc:
            wl["cs_target"] = (random_q(rm, 4, seed=13).astype(np.float32), (np.arange(B) % 4).astype(np.int32))
        return wl
    if name in ("franka_mpc_knots_1024x30_esdf_swept", "franka_mpc_knots_inkernel_1024x30_esdf_swept"):
        # config 4 driven the way the reference's MPC/trajopt drives it: the action is 24 B-spline knots per seed
        # (degree 4, 1 interpolation step -> 30 rows); one C call = knots -> row costs + d cost / d knots
        # (SURVEY.md 8f rank 1: spline evaluated inside the rollout kernel, adjoint kernel right behind it)
        from helpers import random_walk_q
        rm = load_robot("franka")
        B, nk, degree, steps = 1024, 24, 4, 1
        H = (nk + degree + 1) * steps + 1
        knots = random_walk_q(rm, B, nk, seed=300 + seed_offset)
        _, _, gp, gq = O.fk_forward(rm, random_q(rm, B, seed=9))
        goal = (gp[:, :, None, :].copy(), gq[:, :, None, :].copy(), np.arange(B, dtype=np.int32))
        D, S, L = rm.num_dof, rm.num_spheres, rm.num_tool_frames
        bpe = 4 * D * nk / H * 2 + 4 * (S + 1 + 2 * L + D) + 16 * S * 7 + 4 * 4 * D * 2   # knots in / grad out, 4 row grads w+r
        z = np.zeros((B, D), np.float32)
        return dict(robot=rm, cfg=RolloutConfig.trajopt(), B=B, H=H, q=None, goal=goal, cuboid=None,
                    voxel=dict(n=256, voxel=0.01, boxes=12, seed=0), bytes_per_eval=bpe,
                    knots=dict(knots=knots, start=(knots[:, 0].copy(), z, z, z), goal=(knots[:, -1].copy(), z, z, z),
                               dt=np.full(B, 0.05, np.float32), degree=degree, steps=steps, in_kernel="inkernel" in name))
    raise ValueError(f"unknown workload {name}")


def build_engine(wl, device):
    import torch
    from curobo_b200.rollout import RolloutEngine
    from curobo_b200.scene import CuboidData, VoxelData
    from curobo_b200.world import make_box_esdf
    cub = CuboidData.from_world(wl["cuboid"], device) if wl["cuboid"] is not None else None
    vox = None
    if wl["voxel"] is not None:
        v = wl["voxel"]
        sdf = make_box_esdf(n=v["n"], voxel_size=v["voxel"], num_boxes=v["boxes"], seed=v["seed"], xp=torch)
        t = lambda a, dt: torch.as_tensor(np.asarray(a, dtype=dt)).to(device)  # noqa: E731
        vox = VoxelData(t([[[v["n"], v["n"], v["n"], v["voxel"]]]], np.float32), t([[[0, 0, 0, 1, 0, 0, 0, 0]]], np.float32),
                        torch.ones((1, 1), dtype=torch.uint8, device=device), torch.ones(1, dtype=torch.int32, device=device),
                        sdf.reshape(1, 1, -1).contiguous().to(device), 1, 1, 100.0)
    # static synthetic ESDF: the exact lower-bound level is built once (refresh_world) and stays fresh; discrete mode only
    eng = RolloutEngine(wl["robot"], wl["cfg"], device, cub, vox, use_voxel_mip=vox is not None and not wl["cfg"].use_sweep)
    if wl["goal"] is not None:
        gp, gq, idx = wl["goal"]
        eng.update_goal(torch.as_tensor(gp).to(device), torch.as_tensor(gq).to(device), torch.as_tensor(idx).to(device))
    if wl.get("cs_target") is not None:
        tgt, tidx = wl["cs_target"]
        eng.update_cspace_target(torch.as_tensor(tgt).to(device), torch.as_tensor(tidx).to(device))
    if wl.get("dynamics"):
        from curobo_b200.dynamics import Dynamics
        rm = wl["robot"]
        rng = np.random.default_rng(7)
        mc = np.concatenate([rng.uniform(-0.05, 0.05, (rm.num_links, 3)), rng.uniform(0.2, 3.0, (rm.num_links, 1))], 1)
        inn = np.zeros((rm.num_links, 8))
        inn[:, :3] = rng.uniform(0.002, 0.01, (rm.num_links, 3))
        eng.attach_dynamics(Dynamics(rm, mc, inn, device=device), fused=wl["dynamics"] == "fused")
    return eng


def ik_solve_bench(device, problems=512, seeds=32, iters=100, repeats=5):
    """A complete batched IK solve through the public pieces (SURVEY.md 8f rank 2): LBFGSOpt (lbfgs_ik.yml settings:
    history 7, line-search scales [0, .1, .5, 1], approx Wolfe, 100 iterations) driving RolloutEngine.evaluate_action
    on problems x seeds x 4 rows of the config-2 cuboid world -- 3 kernel launches per iteration.  Goals are poses of
    random collision-unchecked configurations; success = best seed within 5 mm and 0.05 rad of the goal."""
    import torch
    from curobo_b200.kinematics import Kinematics
    from curobo_b200.optim import LBFGSOpt, LBFGSOptCfg
    from helpers import random_q
    from oracle import rollout_oracle as O
    wl = make_workload("franka_ik_512x32_cuboid")
    rm, n = wl["robot"], 4
    B, D = problems * seeds, rm.num_dof
    q_goal = random_q(rm, problems, seed=11) * 0.8
    _, _, gp, gq = O.fk_forward(rm, q_goal)
    wl = dict(wl, goal=(gp[:, :, None, :].copy(), gq[:, :, None, :].copy(),
                        np.repeat(np.arange(B) // seeds, n).astype(np.int32)))
    eng = build_engine(wl, device)

    def cost_grad(x):
        out = eng.evaluate_action(x.view(B * n, 1, D))
        return out.cost.view(-1), out.grad_q.view(B * n, D)

    td = lambda a: torch.as_tensor(a).to(device)  # noqa: E731
    opt = LBFGSOpt(LBFGSOptCfg(num_iters=iters), B, 1, D, td(rm.position_limits[0]), td(rm.position_limits[1]), cost_grad, device)
    x0 = td(random_q(rm, B, seed=12))
    opt.optimize(x0)                                                    # warm-up (allocations, plan caches)
    torch.cuda.synchronize(device)
    t0 = time.perf_counter()
    for _ in range(repeats):
        q_sol = opt.optimize(x0)
    torch.cuda.synchronize(device)
    dt_eager = (time.perf_counter() - t0) / repeats
    opt.optimize_graphed(x0)                                            # capture: the whole solve = one CUDA-graph launch
    torch.cuda.synchronize(device)
    t0 = time.perf_counter()
    for _ in range(repeats):
        q_sol = opt.optimize_graphed(x0)
    torch.cuda.synchronize(device)
    dt = (time.perf_counter() - t0) / repeats
    q_sol = q_sol.view(B, D)
    st = Kinematics(rm, device).compute_kinematics(q_sol.view(B, 1, D))
    pos = st.tool_pose_position.reshape(B, -1, 3)[:, 0].detach().cpu().numpy().reshape(problems, seeds, 3)
    quat = st.tool_pose_quaternion.reshape(B, -1, 4)[:, 0].detach().cpu().numpy().reshape(problems, seeds, 4)
    perr = np.linalg.norm(pos - gp[:, 0][:, None, :], axis=-1)
    dotq = np.abs(np.sum(quat * gq[:, 0][:, None, :], axis=-1)).clip(0, 1)
    rerr = 2.0 * np.arccos(dotq)
    ok = ((perr < 5e-3) & (rerr < 0.05)).any(axis=1)
    return {"problems": problems, "seeds": seeds, "iterations": iters, "line_search_candidates": n,
            "launches_per_iteration": 3, "solve_ms": dt * 1e3, "solve_ms_eager_python_loop": dt_eager * 1e3,
            "schedule": "LBFGSOpt.optimize_graphed: initial evaluation + 100 iterations replayed as ONE CUDA graph",
            "ik_solves_per_s": problems / dt,
            "rollout_evals_per_s": B * n * (iters + 1) / dt, "success_rate": float(ok.mean()),
            "median_position_error_mm": float(np.median(perr.min(axis=1)) * 1e3), "timer": "wall clock around the call"}


# ------------------------------------------------------------------------------------------------
# clocks sampling during the timed region
# ------------------------------------------------------------------------------------------------
def rnea_bench(device, peak, cases=(("franka", 16384), ("franka", 30720), ("g1_29", 30720)), iters=20):
    """SURVEY.md 8f rank 3: RNEA inverse dynamics + adjoint over (seed x waypoint) rows, through the backend module
    (C ABI). Inputs resident in HBM, a 160 MB write between iterations flushes L2, CUDA events on the launching stream.
    Inertial parameters are synthetic (random, physically plausible); the kinematic trees are the real robots'."""
    import torch
    from curobo_b200.backends import dynamics as dynamics_cu
    from curobo_b200.dynamics import tree_levels
    from curobo_b200.robot_model import load_robot
    out = {}
    flush = torch.zeros(160 * 1024 * 1024 // 4, device=device)
    t = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a, dtype=dt)).to(device)  # noqa: E731
    for robot, B in cases:
        rm = load_robot(robot)
        nl, D = rm.num_links, rm.num_dof
        rng = np.random.default_rng(7)
        mc = np.concatenate([rng.uniform(-0.05, 0.05, (nl, 3)), rng.uniform(0.2, 3.0, (nl, 1))], 1)
        inn = np.zeros((nl, 8))
        inn[:, :3] = rng.uniform(0.002, 0.01, (nl, 3))
        starts, order = tree_levels(rm.link_map)
        model = (t(rm.fixed_transforms, np.float32), t(mc, np.float32), t(inn, np.float32), t(rm.joint_map_type, np.int8),
                 t(rm.joint_map, np.int16), t(rm.link_map, np.int16), t(rm.joint_offset_map, np.float32),
                 t([0, 0, 0, 0, 0, 9.81], np.float32), t(starts, np.int16), t(order, np.int16))
        nlev = len(starts) - 1
        q, qd, qdd, gt = (t(rng.uniform(-1.5, 1.5, (B, D)), np.float32) for _ in range(4))
        tau = torch.zeros((B, D), device=device)
        cache = torch.zeros((B, nl * 20), device=device)
        g = [torch.zeros((B, D), device=device) for _ in range(3)]
        fwd = lambda: dynamics_cu.launch_rnea_forward(tau, q, qd, qdd, *model, cache, B, nl, D, nlev)  # noqa: E731
        bwd = lambda: dynamics_cu.launch_rnea_backward(*g, gt, q, qd, *model, cache, B, nl, D, nlev)  # noqa: E731
        res = {}
        for name, fn, nbytes in (("forward", fwd, B * 4 * (4 * D + nl * 20)), ("backward", bwd, B * 4 * (6 * D + nl * 20))):
            for _ in range(3):
                fn()
            ts = []
            for _ in range(iters):
                flush.add_(1.0)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
            ms = float(np.median(ts))
            res[name] = {"kernel_ms": ms, "rows_per_s": B / (ms * 1e-3), "bytes_per_row": nbytes // B,
                         "hbm_frac": nbytes / (ms * 1e-3) / 1e9 / peak}
        out[f"{robot}_{B}"] = res
    return out


def edt_bench(device, peak, n=256, iters=10):
    """SURVEY.md 8f rank 4: exact nearest-site transform of an n^3 grid (box shells + sparse noise as sites) through the
    backend module, in place; algorithmic traffic = 3 passes x (4 B read + 4 B write) per voxel; the grid is re-seeded (one
    device copy, outside the timed region) before every iteration; n^3 x 4 B = 64 MiB at n = 256, so every pass streams HBM."""
    import torch
    from curobo_b200.esdf import ParallelBandingEDT, seed_sites_from_occupancy
    g = torch.Generator(device="cpu").manual_seed(0)
    occ = torch.rand((n, n, n), generator=g) < 2e-4
    for lo, hi in (((40, 60, 30), (120, 140, 90)), ((150, 30, 100), (220, 110, 200))):
        box = torch.zeros_like(occ)
        box[lo[0]:hi[0], lo[1]:hi[1], lo[2]:hi[2]] = True
        box[lo[0] + 1:hi[0] - 1, lo[1] + 1:hi[1] - 1, lo[2] + 1:hi[2] - 1] = False
        occ |= box
    fresh = seed_sites_from_occupancy(occ.to(device))
    work = fresh.clone()
    edt = ParallelBandingEDT((n, n, n), 0.01, torch.device(device))
    ts = []
    for i in range(iters + 2):
        work.copy_(fresh)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        edt.propagate(work)
        e1.record()
        torch.cuda.synchronize()
        if i >= 2:
            ts.append(e0.elapsed_time(e1))
    ms = float(np.median(ts))
    nbytes = 3 * 8 * n ** 3
    out = {"grid": [n, n, n], "sites": int(occ.sum()), "transform_ms": ms, "voxels_per_s": n ** 3 / (ms * 1e-3),
           "bytes_per_voxel": 24, "hbm_frac": nbytes / (ms * 1e-3) / 1e9 / peak, "launches": 3,
           "esdf_builder": esdf_builder_bench(device, n)}
    try:
        out["depth_to_esdf"] = depth_to_esdf_bench(device, n)
    except Exception as ex:                                               # noqa: BLE001
        out["depth_to_esdf"] = {"error": repr(ex)[:200]}
    return out


def depth_to_esdf_bench(device, n=256, iters=10, hw=(480, 640)):
    """Depth frame -> collision-ready ESDF (SURVEY.md 8f rank 4, whole chain): DenseTSDF.integrate (two rendered depth images of a
    sphere) -> combined SDF -> DenseESDFBuilder.compute (seed + exact transform + signed fp16 distance); 7 launches per frame."""
    import torch
    from curobo_b200.esdf import DenseESDFBuilder, DenseTSDF
    from curobo_b200.world import depth_scene
    voxel = 2.56 / n
    trunc = 4 * voxel
    K, pos, quat, depth, _ = depth_scene((n, n, n), voxel, n_cam=2, hw=hw, seed=1)
    T = lambda a: torch.as_tensor(np.ascontiguousarray(a)).to(device)  # noqa: E731
    d, k, p, q = T(depth), T(K), T(pos), T(quat)
    tsdf = DenseTSDF((n, n, n), voxel, trunc, device, depth_min=0.05, depth_max=10.0, minimum_tsdf_weight=0.5)
    b = DenseESDFBuilder((n, n, n), voxel, trunc, device)
    ts, ti = [], []
    for i in range(iters + 2):
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record()
        tsdf.integrate(d, k, p, q)
        e1.record()
        b.compute(tsdf.combined_sdf(), None)
        e2.record()
        torch.cuda.synchronize()
        if i >= 2:
            ti.append(e0.elapsed_time(e1))
            ts.append(e0.elapsed_time(e2))
    return {"frame_ms": float(np.median(ts)), "integrate_ms": float(np.median(ti)), "cameras": 2, "image": list(hw),
            "observed_frac": float((tsdf.block_data[..., 1] > 0).float().mean()),
            "stages": "depth integration + combined SDF + seed + 3-pass transform + signed fp16 distance"}


def esdf_builder_bench(device, n=256, iters=10):
    """The whole producer side of the ESDF wire format (SURVEY.md 8f rank 4): dense SDF -> seed sites -> exact transform ->
    signed fp16 distance (curobo_b200.esdf.DenseESDFBuilder = _compute_esdf_impl's three stages), 5 launches."""
    import torch
    from curobo_b200.esdf import DenseESDFBuilder
    from curobo_b200.world import make_box_esdf
    voxel = 2.56 / n                                      # the same 2.56 m world at every grid size
    sdf = make_box_esdf(n=n, voxel_size=voxel, num_boxes=12, seed=0, xp=torch).to(torch.float32).reshape(n, n, n).to(device)
    trunc = 4 * voxel
    sdf = sdf.clamp(-trunc, trunc).contiguous()
    b = DenseESDFBuilder((n, n, n), voxel, trunc, device)
    ts = []
    for i in range(iters + 2):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.compute(sdf, sdf)
        e1.record()
        torch.cuda.synchronize()
        if i >= 2:
            ts.append(e0.elapsed_time(e1))
    ms = float(np.median(ts))
    return {"build_ms": ms, "voxels_per_s": n ** 3 / (ms * 1e-3), "stages": "seed + 3-pass transform + signed fp16 distance",
            "sites": int((b.site_index >= 0).sum())}


class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.samples, self.proc, self.thread, self.idx = [], None, None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "100"], stdout=subprocess.PIPE, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(workload: str):
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(workload)
        except Exception:
            return None
    return None


# ------------------------------------------------------------------------------------------------
# CPU baseline: the numpy oracle on a bounded sample of the same workload
# ------------------------------------------------------------------------------------------------
_ORACLE_CACHE = {}


def _oracle_eval(args):
    wl_name, lo, hi = args
    from oracle import rollout_oracle as O
    if wl_name not in _ORACLE_CACHE:                          # built once in the parent; forked workers inherit it
        _ORACLE_CACHE[wl_name] = (make_workload(wl_name), {})
    wl, extra_cache = _ORACLE_CACHE[wl_name]
    vox = extra_cache.get("vox")
    if wl["voxel"] is not None and vox is None:
        from curobo_b200.world import VoxelWorld, make_box_esdf
        v = wl["voxel"]
        n = 64                                               # same world, coarser grid: the CPU arm's cost is sphere math
        sdf = make_box_esdf(n=n, voxel_size=v["voxel"] * v["n"] / n, num_boxes=v["boxes"], seed=v["seed"])
        vox = VoxelWorld.from_grid(sdf.reshape(n, n, n), v["voxel"] * v["n"] / n)
        extra_cache["vox"] = vox
    q = wl["q"][lo:hi]
    kw = {}
    if wl["goal"] is not None:
        gp, gq, idx = wl["goal"]
        kw = dict(goal_pos=gp, goal_quat=gq, idxs_goal=idx[lo:hi])
    for k, v in wl.get("extra", {}).items():
        kw[k] = v[lo:hi]
    if wl.get("cs_target") is not None:
        kw.update(cspace_target=wl["cs_target"][0], idxs_cspace_target=wl["cs_target"][1][lo:hi])
    t0 = time.perf_counter()
    O.rollout_cost_grad(wl["robot"], q, wl["cfg"].to_oracle_cfg(wl["robot"].num_tool_frames), world_cuboid=wl["cuboid"],
                        world_voxel=vox, **kw)
    return time.perf_counter() - t0


def cpu_baseline(wl_name: str, target_seconds: float = 12.0, procs: int = 1):
    """evals/s of the oracle port.  procs == 1: single numpy process; procs > 1: one process per host core,
    each evaluating its own slice of the sample."""
    wl = make_workload(wl_name)
    probe = 64
    t = _oracle_eval((wl_name, 0, probe))
    t = _oracle_eval((wl_name, 0, probe))                    # warm caches / imports
    per_eval = t / probe
    n = int(max(probe, min(wl["B"], target_seconds / per_eval)))
    if procs <= 1:
        dt = _oracle_eval((wl_name, 0, n))
        return n / dt, 1, f"{n} of {wl['B'] * wl['H']} evals of {wl_name}, numpy oracle, 1 process"
    import multiprocessing as mp
    n = int(min(wl["B"], n * procs)) // procs * procs
    chunk = n // procs
    with mp.get_context("fork").Pool(procs) as pool:
        t0 = time.perf_counter()
        pool.map(_oracle_eval, [(wl_name, i * chunk, (i + 1) * chunk) for i in range(procs)])
        dt = time.perf_counter() - t0
    return n / dt, procs, f"{n} of {wl['B'] * wl['H']} evals of {wl_name}, numpy oracle, {procs} processes"


def measured_swept_samples(wl_name: str, seeds: int = 6):
    """Mean number of ESDF samples per (sphere, waypoint) of a swept workload (SURVEY.md 8d: "n_s in [1, 7], report the measured
    mean"): the oracle's adaptive sweep counted on the first `seeds` trajectories of the workload against the same analytic world
    (128^3 instead of 256^3: the sample count depends on the geometry, not on the grid pitch)."""
    from curobo_b200.world import VoxelWorld, make_box_esdf
    from oracle import rollout_oracle as O
    wl = make_workload(wl_name)
    if wl.get("q") is None or wl["voxel"] is None:
        return None
    v, n = wl["voxel"], 128
    sdf = make_box_esdf(n=n, voxel_size=v["voxel"] * v["n"] / n, num_boxes=v["boxes"], seed=v["seed"])
    vox = VoxelWorld.from_grid(np.asarray(sdf).reshape(n, n, n), v["voxel"] * v["n"] / n)
    q = wl["q"][:seeds]
    B, H, D = q.shape
    _, sph, _, _ = O.fk_forward(wl["robot"], q.reshape(B * H, D))
    stats = {}
    O.scene_collision(sph.reshape(B, H, -1, 4), 1.0, wl["cfg"].scene_activation, None, vox, None, sweep=True, stats=stats)
    return stats["samples"] / max(1, stats["sphere_obstacle_pairs"])


# ------------------------------------------------------------------------------------------------
def workload_config(name, wl):
    """The `config` object -- identical in both arms (the driver compares them)."""
    return {"workload": name, "robot": wl["robot"].name, "batch_per_gpu": wl["B"], "horizon": wl["H"],
            "evals_per_step_per_gpu": wl["B"] * wl["H"],
            "world": "cuboids" if wl["cuboid"] is not None else "esdf_256^3_fp16",
            "cache": "GPU arm: L2 flushed (256 MiB write) between timed steps", "timer": "GPU arm: cuda events per step, max over ranks"}


def _limit_blas_threads():
    """One BLAS / OpenMP thread per worker process: 128 forked numpy workers each spinning up a 128-thread pool is what made the
    CPU arm swing 4x between boxes in round 1."""
    for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
        os.environ[k] = "1"
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(1)
    except Exception:                                                     # noqa: BLE001
        pass


def run_reference_arm(args):
    """--impl reference: the reference has no CPU implementation of this path (DeviceCfg defaults to cuda,
    kernels are CUDA/Warp only), so the CPU arm is the oracle port (numpy, float32; NOT PyTorch: the port is written in numpy)
    on all host cores, one single-threaded process per core.  Each step evaluates a bounded sample of the workload (one slice
    per core); the whole run is sized to end within ~2 minutes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    _limit_blas_threads()
    cores = os.cpu_count() or 1
    wl = make_workload(args.workload)
    _oracle_eval((args.workload, 0, 64))                       # import + warm caches in the parent (fork shares them)
    per_eval = _oracle_eval((args.workload, 0, 64)) / 64
    budget = max(0.15, min(10.0, 100.0 / max(1, args.steps + args.warmup)))     # seconds of wall time per step
    chunk = int(max(16, min(wl["B"] // cores, budget / per_eval)))
    n = chunk * cores
    vals = []
    with mp.get_context("fork").Pool(cores) as pool:
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            pool.map(_oracle_eval, [(args.workload, c * chunk, (c + 1) * chunk) for c in range(cores)])
            dt = time.perf_counter() - t0
            if i >= args.warmup:
                vals.append(n / dt)
    value = float(np.mean(vals))
    sample = f"{n} of {wl['B'] * wl['H']} evals of {args.workload} per step, numpy (not torch) oracle, {cores} single-threaded processes"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * n / value, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.workload, wl),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def pin_to_gpu_numa_node(local_rank: int):
    """Bind this rank's host threads to the CPUs NVML reports as local to its GPU (GPUs 4-7 sit on NUMA node 1 on the 8-GPU
    boxes; an unpinned rank that lands on the other socket pays a cross-socket hop on every launch and pinned copy)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1]
        cpus = [c for c in cpus if c in os.sched_getaffinity(0)]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:                                                     # noqa: BLE001
        pass
    return 0


def shard_workload(wl, lo, hi):
    """Rows [lo, hi) of a workload (strong scaling: the total is fixed, a rank evaluates its slice)."""
    w = dict(wl)
    w["B"] = hi - lo
    w["q"] = wl["q"][lo:hi]
    if wl["goal"] is not None:
        gp, gq, idx = wl["goal"]
        w["goal"] = (gp, gq, idx[lo:hi].copy())
    if "extra" in wl:
        w["extra"] = {k: v[lo:hi] for k, v in wl["extra"].items()}
    if wl.get("cs_target") is not None:
        w["cs_target"] = (wl["cs_target"][0], wl["cs_target"][1][lo:hi].copy())
    return w


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="franka_ik_512x32_cuboid")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ik-solve", type=int, default=1,
                    help="1: also time a complete 100-iteration L-BFGS IK solve (512 goals x 32 seeds), reported under 'ik_solve'")
    ap.add_argument("--edt", type=int, default=1, help="1: also time the exact nearest-site transform (256^3), reported under 'edt'")
    ap.add_argument("--rnea", type=int, default=1, help="1: also time the RNEA inverse-dynamics kernels, reported under 'rnea'")
    ap.add_argument("--sharded", type=int, default=1,
                    help="1: also strong-scale BASELINE configs 4 and 5 over the N ranks (rollout + sharded solve), under 'sharded'")
    ap.add_argument("--reference-design", type=int, default=1,
                    help="1 (N=1 only): time the reference's own kernels compiled for sm_100a, chained unfused from a CUDA graph "
                         "(scripts/bench_reference_design.py, separate process), under 'reference_design_gpu'")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the headline workload's outputs of its last timed step (the RolloutOutput arrays) as DIR/<name>.npy")
    ap.add_argument("--extra-workloads", default="franka_16384_esdf,franka_trajopt_32x32_esdf_swept,franka_mpc_1024x30_esdf_swept,franka_mpc_knots_1024x30_esdf_swept,franka_mpc_knots_inkernel_1024x30_esdf_swept,g1_29_8192_esdf,g1_43_8192_esdf,franka_mpc_1024x30_esdf_swept_dynamics_host,franka_mpc_1024x30_esdf_swept_dynamics,franka_mpc_knots_1024x30_esdf_swept_dynamics",
                    help="comma list, measured briefly on rank 0 at N=1 and reported under 'other_workloads'")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA GPU: the rollout path has no CPU fallback")
    pinned_cpus = pin_to_gpu_numa_node(local_rank)
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    from curobo_b200.rollout import HostRolloutPipeline
    # clocks are sampled from here to the end of the e2e loop (pre-roll, timed steps, e2e): the timed region alone
    # (K x 77 us) is shorter than nvidia-smi's 100 ms period
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()

    def barrier():
        if world > 1:
            dist.barrier()

    def make_run(wl, eng, q):
        kw = {k: torch.as_tensor(v).to(device) for k, v in wl.get("extra", {}).items()}
        if "knots" in wl:
            from curobo_b200.trajectory import JointState
            kn = wl["knots"]
            td = lambda a: torch.as_tensor(a).to(device)  # noqa: E731
            kq = td(kn["knots"])
            ks = JointState(*[td(x) for x in kn["start"]])
            kg = JointState(*[td(x) for x in kn["goal"]], dt=td(kn["dt"]))
            kidx = torch.arange(wl["B"], dtype=torch.int32, device=device)
            kimp = torch.zeros(wl["B"], dtype=torch.uint8, device=device)
            return (lambda: eng.evaluate_knots(kq, ks, kidx, kg, kidx, kimp, kn["degree"], kn["steps"],
                                               in_kernel_spline=kn["in_kernel"])), kw
        return (lambda: eng.evaluate_action(q, **kw)), kw

    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=device)       # 2x the 126 MB L2

    def timed_steps(run, steps, do_flush):
        stream = torch.cuda.current_stream(device)
        starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        barrier()
        torch.cuda.synchronize(device)
        for i in range(steps):
            if do_flush:
                flush.fill_(i & 0xFF)                       # evict L2 between timed steps (outside the event pair)
            starts[i].record(stream)
            run()
            ends[i].record(stream)
        torch.cuda.synchronize(device)
        barrier()
        return [s.elapsed_time(e) for s, e in zip(starts, ends)]

    def timed_run(wl_or_name, steps, warmup, preroll_s=0.0, warm_too=False):
        wl = make_workload(wl_or_name, seed_offset=rank) if isinstance(wl_or_name, str) else wl_or_name
        eng = build_engine(wl, device)
        q = torch.as_tensor(wl["q"]).to(device) if wl.get("q") is not None else None
        run, kw = make_run(wl, eng, q)
        for _ in range(warmup):
            run()
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        while time.perf_counter() - t0 < preroll_s:          # untimed pre-roll: clocks settle, the sampler gets samples under load
            for _ in range(50):
                run()
            torch.cuda.synchronize(device)
        ms = timed_steps(run, steps, True)
        ms_warm = timed_steps(run, steps, False) if warm_too else None
        wl["kw"] = kw
        return wl, eng, q, ms, ms_warm

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    if "knots" in args.workload:
        raise SystemExit("the B-spline knots workload is measured under other_workloads (--extra-workloads) only")
    def last_kernel():
        """name of the kernel the last rollout launch used (include/curobo_b200.h: CB200_VARIANT_*)"""
        from curobo_b200 import lib as cblib
        names = {1: "rollout_fused_kernel", 2: "rollout_fused_kernel (80-register arm build)", 4: "rollout_fused_big_kernel",
                 5: "rollout_fused_team_kernel<2 warps per row>", 6: "rollout_fused_team_kernel<4 warps per row>",
                 7: "rollout_traj_kernel", 8: "rollout_traj_dyn_kernel", 9: "rollout_tile_kernel", 10: "rollout_lane_kernel"}
        return names.get(int(cblib.load().cb200_last_rollout_variant()), "?")

    wl, eng, q, ms_list, ms_warm = timed_run(args.workload, args.steps, args.warmup, preroll_s=0.5, warm_too=True)
    headline_kernel = last_kernel()
    if args.dump_outputs and rank == 0:
        dump_outputs(eng.out, args.dump_outputs)             # before the e2e pipeline below reuses `eng`
    evals_per_step = wl["B"] * wl["H"]
    total_ms_max = max_over_ranks(float(sum(ms_list)))
    value = world * evals_per_step * args.steps / (total_ms_max * 1e-3)
    value_warm = world * evals_per_step * args.steps / (max_over_ranks(float(sum(ms_warm))) * 1e-3)

    # ---- e2e: what a user of the public API does per optimizer iteration with HOST data: pinned host q -> H2D ->
    # RolloutEngine.evaluate_action -> D2H of cost + grad_q, through curobo_b200.rollout.HostRolloutPipeline: every step is ONE
    # CUDA-graph launch (copy, kernel, copies) on one of two slots (two streams, two engines = two buffer sets), so step
    # i+1's upload overlaps step i's kernel.  Every step's copies are inside the timed region.
    D = wl["robot"].num_dof
    pipe = HostRolloutPipeline([eng, build_engine(wl, device)], wl["B"], wl["H"], **wl["kw"])
    for sl in pipe.slots:
        sl.q_host.copy_(torch.as_tensor(wl["q"]))
    for i in range(4):
        pipe.submit(i & 1)
    pipe.wait_all()
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        pipe.submit(i & 1)
    pipe.wait_all()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
    e2e_value = world * evals_per_step * args.steps / (e2e_ms * 1e-3)
    h2d, d2h = pipe.h2d_bytes, pipe.d2h_bytes
    # sanity: the host copy of the last step's result is the device result
    last = pipe.slots[(args.steps - 1) & 1]
    assert torch.equal(last.cost_host, last.engine.out.cost.cpu())
    clocks = sampler.stop() if sampler else None

    # ---- BASELINE configs 4 and 5, strong-scaled over the ranks: total rows fixed, this rank evaluates rows / N.
    # (a) rollout only: K2 timed steps (events, L2 flushed), max over ranks; (b) a complete seed-sharded solve through
    # curobo_b200.sharded.ShardedSolver: per-rank L-BFGS (one CUDA graph) + the end-of-solve all_gather, all inside the timed region.
    sharded = {}
    if args.sharded:
        from curobo_b200.optim import LBFGSOptCfg
        from curobo_b200.sharded import ShardedSolver, shard_rows
        for key, name, max_world, iters in (("config5_g1_29_8192_esdf", "g1_29_8192_esdf", 8, 20),
                                            ("config4_franka_mpc_1024x30", "franka_mpc_1024x30_esdf_swept", 4, 10)):
            if world > max_world:
                sharded[key] = {"skipped": f"BASELINE shards this config over at most {max_world} GPUs"}
                continue
            try:
                full = make_workload(name)
                lo, hi = shard_rows(full["B"], rank, world)
                part = shard_workload(full, lo, hi)
                k2 = max(5, min(50, args.steps))
                w2, e2, _, ms2, _ = timed_run(part, k2, 3)
                roll_ms = max_over_ranks(float(np.mean(ms2)))
                res = {"total_rows": full["B"], "horizon": full["H"], "rows_per_gpu": hi - lo,
                       "rollout_ms_per_step": roll_ms, "rollout_evals_per_s": full["B"] * full["H"] / (roll_ms * 1e-3)}
                # the solve: every seed's waypoint positions are the optimisation variable, 4 line-search candidates per seed
                cfg_o = LBFGSOptCfg(num_iters=iters)
                n = len(cfg_o.line_search_scale)
                rep = lambda a: np.repeat(a, n, axis=0)  # noqa: E731
                cand = dict(part, B=part["B"] * n, q=rep(part["q"]))
                if part["goal"] is None:
                    # whole-body IK: every seed pulls the robot's tool frames towards the poses of one reference posture
                    from curobo_b200.rollout import RolloutConfig
                    from helpers import humanoid_q
                    from oracle import rollout_oracle as O
                    _, _, gp, gq = O.fk_forward(full["robot"], humanoid_q(full["robot"], 1, seed=77, scale=0.5))
                    part = dict(part, goal=(gp[:, :, None, :].copy(), gq[:, :, None, :].copy(), np.zeros(part["B"], np.int32)))
                    cand["cfg"] = RolloutConfig(**{**part["cfg"].__dict__, "pose_weight": (2000.0, 100.0)})
                if part["goal"] is not None:
                    cand["goal"] = (part["goal"][0], part["goal"][1], rep(part["goal"][2]))
                if part.get("cs_target") is not None:
                    cand["cs_target"] = (part["cs_target"][0], rep(part["cs_target"][1]))
                cand.pop("extra", None)                           # vel / acc / jerk: finite differences inside the kernel
                eng_s = build_engine(cand, device)
                kw_s = {}
                if full["H"] > 1:
                    kw_s["dt"] = torch.full((cand["B"],), 0.05, device=device)
                solver = ShardedSolver(eng_s, full["B"], full["H"], cfg_o, eval_kwargs=kw_s)
                x0 = torch.as_tensor(part["q"]).to(device)
                solver.solve(x0)                                  # warm-up + graph capture
                torch.cuda.synchronize(device)
                ts = []
                for _ in range(3):
                    barrier()
                    torch.cuda.synchronize(device)
                    t0 = time.perf_counter()
                    cost_all, best_row, _ = solver.solve(x0)
                    torch.cuda.synchronize(device)
                    ts.append(max_over_ranks((time.perf_counter() - t0) * 1e3))
                sm = float(np.median(ts))
                res.update({"solve_ms": sm, "solve_iterations": iters, "line_search_candidates": n,
                            "solve_rollout_evals_per_s": full["B"] * full["H"] * n * (iters + 1) / (sm * 1e-3),
                            "solve_includes": "per-rank L-BFGS (one CUDA graph) + all_gather of seed costs + best action",
                            "best_row": int(best_row), "best_cost": float(cost_all[best_row])})
                sharded[key] = res
                del solver, eng_s, e2
            except Exception as ex:                                               # noqa: BLE001
                sharded[key] = {"error": repr(ex)[:300]}

    if rank == 0:
        peak, peak_src = measured_hbm_peak()
        kernel_ms = float(np.mean(ms_list))
        achieved = wl["bytes_per_eval"] * evals_per_step / (kernel_ms * 1e-3) / 1e9
        cfg_obj = workload_config(args.workload, wl)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": cfg_obj,
            "sharding": f"seeds x{world} (no data-path collective); ranks pinned to their GPU's NUMA cpus: {pinned_cpus}",
            "value_warm_l2": value_warm,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "cache": "no flush (inputs arrive by H2D every step); compare with value_warm_l2",
                    "api": "curobo_b200.rollout.HostRolloutPipeline: one CUDA graph per step = H2D + rollout kernel + D2H"},
            "gpu_launches": args.steps,
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": headline_kernel, "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": ncu_traffic(args.workload),
                         "bytes_per_eval": wl["bytes_per_eval"], "kernel_ms": kernel_ms, "peak_source": peak_src,
                         "note": "path is FP32-issue/latency bound by construction (working set is L2-resident); see DESIGN.md"},
            "sharded": sharded,
        }
        others = {}
        if world == 1:

            def extra(name):
                try:
                    w2, _, _, ms2, _ = timed_run(name, max(5, args.steps // 5), 3)
                    k_ms = float(np.mean(ms2))
                    ach = w2["bytes_per_eval"] * w2["B"] * w2["H"] / (k_ms * 1e-3) / 1e9
                    others[name] = {"value": w2["B"] * w2["H"] / (k_ms * 1e-3), "kernel_ms": k_ms, "kernel": last_kernel(),
                                    "bytes_per_eval": w2["bytes_per_eval"], "hbm_frac": ach / peak}
                    if w2["cfg"].use_sweep and w2.get("q") is not None and name in ("franka_mpc_1024x30_esdf_swept",
                                                                                     "franka_trajopt_32x32_esdf_swept"):
                        ns = measured_swept_samples(name)       # bytes_per_eval above bounds n_s with 7; this is the measured mean
                        if ns is not None:
                            S_ = w2["robot"].num_spheres
                            bpe_m = w2["bytes_per_eval"] - 16 * S_ * 7 + 16 * S_ * ns
                            others[name].update({"n_s_mean_measured": ns, "bytes_per_eval_measured": bpe_m,
                                                 "hbm_frac_measured": bpe_m * w2["B"] * w2["H"] / (k_ms * 1e-3) / 1e9 / peak})
                except Exception as ex:                                           # noqa: BLE001
                    others[name] = {"error": repr(ex)[:200]}

            for name in [w for w in args.extra_workloads.split(",") if w]:
                extra(name)
            line["other_workloads"] = others
            if args.ik_solve:
                try:
                    line["ik_solve"] = ik_solve_bench(device)
                except Exception as ex:                                               # noqa: BLE001
                    line["ik_solve"] = {"error": repr(ex)[:200]}
            if args.rnea:
                try:
                    line["rnea"] = rnea_bench(device, peak)
                except Exception as ex:                                               # noqa: BLE001
                    line["rnea"] = {"error": repr(ex)[:200]}
            if args.edt:
                try:
                    line["edt"] = edt_bench(device, peak)
                except Exception as ex:                                               # noqa: BLE001
                    line["edt"] = {"error": repr(ex)[:200]}
            if args.reference_design:
                line["reference_design_gpu"] = reference_design_leg()
            if not args.no_cpu_baseline:
                _limit_blas_threads()
                v, cores, sample = cpu_baseline(args.workload, target_seconds=12.0, procs=1)
                line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}
        # compact, LAST: BASELINE.json configs on one short object (the driver keeps the tail of the line)
        bc = {"c2_franka_ik_512x32_cuboid": {"evals_per_s": round(value), "ms": round(kernel_ms, 4), "e2e_evals_per_s": round(e2e_value)}}
        for key, name in (("c3_franka_trajopt_32x32_esdf", "franka_trajopt_32x32_esdf_swept"),
                          ("c4_franka_mpc_1024x30_esdf", "franka_mpc_1024x30_esdf_swept"), ("c5_g1_29_8192_esdf", "g1_29_8192_esdf")):
            if name in others and "value" in others[name]:
                bc[key] = {"evals_per_s": round(others[name]["value"]), "ms": round(others[name]["kernel_ms"], 4)}
        for key, short in (("config4_franka_mpc_1024x30", "c4_sharded"), ("config5_g1_29_8192_esdf", "c5_sharded")):
            r = sharded.get(key, {})
            if "rollout_evals_per_s" in r:
                bc[short] = {"n": world, "evals_per_s": round(r["rollout_evals_per_s"]), "ms": round(r["rollout_ms_per_step"], 4),
                             "solve_ms": round(r.get("solve_ms", 0.0), 3)}
        rd = line.get("reference_design_gpu")
        if isinstance(rd, dict) and "workloads" in rd:
            bc["ref_design_gpu_ms"] = {k: round(v["reference_design_ms"], 4) for k, v in rd["workloads"].items()}
        if "ik_solve" in line and "solve_ms" in line["ik_solve"]:
            bc["ik_solve_ms"] = round(line["ik_solve"]["solve_ms"], 3)
        line["baseline_configs"] = bc
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out, directory, cap_bytes=64 << 20):
    """Every array of a RolloutOutput as <directory>/<field>.npy: float32 as computed, integer fields as float64 (exact).
    Above cap_bytes in all, every array keeps the same fixed seeded sample of its rows (leading axis), listed in rows.npy."""
    import dataclasses
    import torch
    arrays = {f.name: getattr(out, f.name) for f in dataclasses.fields(out)}
    arrays = {k: v.detach().cpu().numpy() for k, v in arrays.items() if torch.is_tensor(v)}
    arrays = {k: v if v.dtype in (np.float32, np.float64) else v.astype(np.float64) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    if total > cap_bytes:
        n = next(iter(arrays.values())).shape[0]
        rows = np.sort(np.random.default_rng(0).choice(n, max(1, n * cap_bytes // total - 1), replace=False))
        arrays = {k: v[rows] for k, v in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    os.makedirs(directory, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(directory, f"{k}.npy"), v)


def reference_design_leg():
    """The kernel to beat, on the same GPU: the reference's own CUDA kernels (compiled for sm_100a under oracle/_ref) chained
    unfused with stand-alone scene / pose / c-space kernels and replayed from a CUDA graph (scripts/bench_reference_design.py).
    Runs in its own process -- the product path in this process never loads oracle/_ref."""
    try:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "bench_reference_design.py"), "--json"],
                           capture_output=True, text=True, timeout=600)
        for ln in reversed(r.stdout.strip().splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)
        return {"error": (r.stderr or r.stdout)[-300:]}
    except Exception as ex:                                                       # noqa: BLE001
        return {"error": repr(ex)[:200]}


if __name__ == "__main__":
    main()
