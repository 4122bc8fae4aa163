"""GPU parity of the B-spline knot -> state kernels and their adjoint (SURVEY.md 8f rank 1), called through the C ABI
(curobo_b200.backends.trajectory), against
  * the numpy oracle (oracle/bspline_oracle.py), and
  * the REFERENCE's own kernels (same nvcc flags; their outputs on these inputs recorded on a B200, tests/ref_kernels.py): forward and adjoint
    are expected to agree to float rounding of identically ordered arithmetic -> tolerance 2 ulp-ish (rtol 1e-6),
    and bit-exact for the adjoint with power-of-two interpolation steps where the summation order is reproduced.
Tolerances vs the oracle (numpy divides exactly, the kernels use --prec-div=false): rel 2e-5 of the output scale.
"""
import numpy as np
import pytest
import torch

import ref_kernels
from bspline_cases import CASES, case_id, make_case
from curobo_b200.backends import trajectory as trajectory_cu
from curobo_b200.trajectory import (BSplineIdxKernel, ControlSpace, JointState, StateFromBSplineKnot,
                                    get_bspline_interpolation)
from oracle import bspline_oracle as bo

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def T(a, dt=None):
    t = torch.as_tensor(np.ascontiguousarray(a)).to(DEV)
    return t.to(dt) if dt is not None else t


def dev_case(c):
    d = dict(c)
    d["knots_t"] = T(c["knots"])
    d["start_t"] = tuple(T(x) for x in c["start"])
    d["goal_t"] = tuple(T(x) for x in c["goal"])
    d["sidx_t"], d["gidx_t"] = T(c["start_idx"]), T(c["goal_idx"])
    d["dt_t"], d["imp_t"] = T(c["traj_dt"]), T(c["implicit"])
    d["grads_t"] = tuple(T(g) for g in c["grads"])
    return d


def time_major(outs):
    """[B,T,D] states -> [T,B,D] (few seeds, many waypoints: the recorded sample keeps whole waypoints, first and last
    included), the per-seed dt as it is."""
    return [o.transpose(0, 1) for o in outs[:4]] + list(outs[4:])


def ours_forward(c):
    B, Tn, D = c["B"], c["T"], c["D"]
    outs = [torch.full((B, Tn, D), float("nan"), device=DEV) for _ in range(4)]
    odt = torch.zeros((B,), device=DEV)
    trajectory_cu.launch_bspline_interpolation_forward_kernel(
        *outs, odt, c["knots_t"], *c["start_t"], *c["goal_t"], c["sidx_t"], c["gidx_t"], c["dt_t"], c["imp_t"], B, Tn, D,
        c["nk"], c["degree"])
    return outs + [odt]


def ours_backward(c):
    out = torch.full((c["B"], c["nk"], c["D"]), float("nan"), device=DEV)
    trajectory_cu.launch_bspline_interpolation_backward_kernel(
        out, *c["grads_t"], c["dt_t"], c["gidx_t"], c["imp_t"], c["B"], c["T"], c["D"], c["nk"], c["degree"])
    return out


@pytest.mark.parametrize("kw", CASES, ids=case_id)
def test_forward_vs_oracle_and_reference(kw):
    c = dev_case(make_case(**kw))
    got = ours_forward(c)
    want = bo.bspline_forward(c["knots"], c["start"], c["goal"], c["start_idx"], c["goal_idx"], c["traj_dt"], c["implicit"],
                              c["T"], c["degree"])
    for k in range(4):
        g, w = got[k].cpu().numpy(), want[k]
        assert np.isfinite(g).all()
        assert np.allclose(g, w, rtol=2e-5, atol=2e-5 * max(1.0, np.abs(w).max())), f"derivative {k} vs oracle"
    assert np.array_equal(got[4].cpu().numpy(), want[4])
    if ref_kernels.comparing():
        ref = ref_kernels.recorded(("bspline", "forward", case_id(kw)), lambda: time_major(ref_kernels.bspline_forward(
            c["knots_t"], c["start_t"], c["goal_t"], c["sidx_t"], c["gidx_t"], c["dt_t"], c["imp_t"], c["T"], c["degree"])))
        for k in range(4):
            g, r = ref.at(k, got[k].cpu().numpy().swapaxes(0, 1)), ref[k]
            assert np.allclose(g, r, rtol=1e-6, atol=1e-6 * max(1.0, np.abs(r).max())), f"derivative {k} vs reference"
        assert np.array_equal(ref.at(4, got[4].cpu().numpy()), ref[4])


@pytest.mark.parametrize("kw", CASES, ids=case_id)
def test_backward_vs_oracle_and_reference(kw):
    c = dev_case(make_case(**kw))
    got = ours_backward(c).cpu().numpy()
    want = bo.bspline_backward(*c["grads"], c["traj_dt"], c["goal_idx"], c["implicit"], c["nk"], c["degree"])
    assert np.allclose(got, want, rtol=1e-4, atol=1e-5 * np.abs(want).max())
    steps = c["steps"]
    if ref_kernels.comparing() and (steps & (steps - 1)) == 0:
        # the reference's shuffle tree is only valid for power-of-two step counts (it mis-pairs lanes otherwise)
        ref = ref_kernels.recorded(("bspline", "backward", case_id(kw)), lambda: ref_kernels.bspline_backward(
            c["grads_t"], c["dt_t"], c["gidx_t"], c["imp_t"], c["nk"], c["degree"]))
        assert np.allclose(ref.at(0, got), ref[0], rtol=1e-6, atol=1e-6 * np.abs(ref[0]).max())


def test_single_dt_vs_oracle_and_reference():
    c = make_case(seed=21, B=6, nk=8, D=7, steps=4, degree=4, implicit=False)
    Tn = 70
    c = dev_case(dict(c, T=Tn))
    interp_h = np.array([52, 39, 69, 13, 200, 26], np.int32)
    out = JointState.zeros((6, Tn, 7), DEV)
    start, goal = JointState(*c["start_t"]), JointState(*c["goal_t"])
    idt = torch.tensor([0.025], device=DEV)
    get_bspline_interpolation(c["knots_t"], None, start, goal, c["sidx_t"], c["gidx_t"], idt, c["imp_t"], T(interp_h), out, 4)
    want = bo.bspline_forward(c["knots"], c["start"], c["goal"], c["start_idx"], c["goal_idx"], c["traj_dt"], c["implicit"],
                              Tn, 4, interpolation_horizon=interp_h, interpolation_dt=np.float32(0.025))
    got = [out.position, out.velocity, out.acceleration, out.jerk]
    for g, w in zip(got, want[:4]):
        assert np.allclose(g.cpu().numpy(), w, rtol=2e-5, atol=2e-5 * max(1.0, np.abs(w).max()))
    if ref_kernels.comparing():
        ref = ref_kernels.recorded(("bspline", "single_dt"), lambda: time_major(ref_kernels.bspline_single_dt(
            c["knots_t"], c["start_t"], c["goal_t"], c["sidx_t"], c["gidx_t"], idt, c["imp_t"], T(interp_h), Tn, 4)))
        for k, g in enumerate(got):
            r = ref[k]
            assert np.allclose(ref.at(k, g.cpu().numpy().swapaxes(0, 1)), r, rtol=1e-6, atol=1e-6 * max(1.0, float(np.abs(r).max())))


@pytest.mark.parametrize("implicit", [False, True])
def test_autograd_function_and_state_transition(implicit):
    """StateFromBSplineKnot.forward + loss.backward(): u_act.grad equals the oracle's adjoint of d loss / d state."""
    B, nk, D, steps = 8, 8, 7, 4
    c = dev_case(make_case(seed=31, B=B, nk=nk, D=D, steps=steps, degree=4, implicit=implicit))
    fn = StateFromBSplineKnot(DEV, D, batch_size=B, n_knots=nk, interpolation_steps=steps,
                              use_implicit_goal_state=implicit, control_space=ControlSpace.BSPLINE_4)
    assert fn.padded_horizon == c["T"]
    start = JointState(*c["start_t"])
    goal = JointState(*c["goal_t"], dt=c["dt_t"])
    out = JointState.zeros((B, c["T"], D), DEV)
    u = c["knots_t"].clone().requires_grad_(True)
    seq = fn.forward(start, u, out, start_state_idx=c["sidx_t"], goal_state=goal, goal_state_idx=c["gidx_t"],
                     use_implicit_goal_state=c["imp_t"])
    w = c["grads_t"]
    loss = (seq.position * w[0]).sum() + (seq.velocity * w[1]).sum() + (seq.acceleration * w[2]).sum() + (seq.jerk * w[3]).sum()
    loss.backward()
    want = bo.bspline_backward(*c["grads"], c["traj_dt"], c["goal_idx"], c["implicit"], nk, 4)
    assert np.allclose(u.grad.cpu().numpy(), want, rtol=1e-4, atol=1e-5 * np.abs(want).max())


def test_error_behaviour():
    c = dev_case(make_case(seed=41, B=2, nk=8, D=7, steps=4, degree=4, implicit=False))
    B, Tn, D = c["B"], c["T"], c["D"]
    outs = [torch.zeros((B, Tn, D), device=DEV) for _ in range(4)]
    odt = torch.zeros((B,), device=DEV)
    args = (*outs, odt, c["knots_t"], *c["start_t"], *c["goal_t"], c["sidx_t"], c["gidx_t"], c["dt_t"], c["imp_t"], B, Tn, D, c["nk"])
    with pytest.raises(RuntimeError, match="Unsupported B-spline degree"):
        trajectory_cu.launch_bspline_interpolation_forward_kernel(*args, 6)
    with pytest.raises(ValueError, match="dtype"):
        bad = list(args)
        bad[5] = c["knots_t"].double()
        trajectory_cu.launch_bspline_interpolation_forward_kernel(*bad, 4)
    with pytest.raises(ValueError, match="CUDA-only|device"):
        bad = list(args)
        bad[5] = c["knots_t"].cpu()
        trajectory_cu.launch_bspline_interpolation_forward_kernel(*bad, 4)
    g = [torch.zeros((B, 5, D), device=DEV) for _ in range(4)]
    out = torch.zeros((B, c["nk"], D), device=DEV)
    with pytest.raises(RuntimeError, match="horizon must be greater than 5"):
        trajectory_cu.launch_bspline_interpolation_backward_kernel(out, *g, c["dt_t"], c["gidx_t"], c["imp_t"], B, 5, D, c["nk"], 4)
    g = [torch.zeros((B, 10, D), device=DEV) for _ in range(4)]
    with pytest.raises(RuntimeError, match="interpolation_steps is 0"):
        trajectory_cu.launch_bspline_interpolation_backward_kernel(out, *g, c["dt_t"], c["gidx_t"], c["imp_t"], B, 10, D, c["nk"], 4)
    # after the rejected launches the library and torch are still healthy
    torch.cuda.synchronize()
    assert torch.isfinite(ours_forward(c)[0]).all()


def test_full_size_adjoint_property_and_graph_capture():
    """MPC / trajopt scale (1024 seeds x 16 knots x 7 dof, 4 steps, degree 4 -> 85 rows): <J du, g> == <du, J^T g> on the
    GPU alone (size-independent property), and both launches are CUDA-graph capturable."""
    B, nk, D, steps, deg = 1024, 16, 7, 4, 4
    c = dev_case(make_case(seed=51, B=B, nk=nk, D=D, steps=steps, degree=deg, implicit=False, mixed_implicit=True))
    base = ours_forward(c)[:4]
    du = torch.randn_like(c["knots_t"])
    c2 = dict(c, knots_t=(c["knots_t"] + du).contiguous())
    pert = ours_forward(c2)[:4]
    lhs = sum(((p.double() - b.double()) * g.double()).sum() for b, p, g in zip(base, pert, c["grads_t"]))
    scale = sum(((p.double() - b.double()) * g.double()).abs().sum() for b, p, g in zip(base, pert, c["grads_t"]))
    gk = ours_backward(c)
    rhs = (gk.double() * du.double()).sum()
    assert abs(float(lhs - rhs)) < 1e-5 * float(scale)

    outs = [torch.zeros_like(base[0]) for _ in range(4)]
    odt = torch.zeros((B,), device=DEV)
    gout = torch.zeros_like(gk)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            trajectory_cu.launch_bspline_interpolation_forward_kernel(
                *outs, odt, c["knots_t"], *c["start_t"], *c["goal_t"], c["sidx_t"], c["gidx_t"], c["dt_t"], c["imp_t"], B,
                c["T"], D, nk, deg)
            trajectory_cu.launch_bspline_interpolation_backward_kernel(
                gout, *c["grads_t"], c["dt_t"], c["gidx_t"], c["imp_t"], B, c["T"], D, nk, deg)
        graph.replay()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    assert torch.equal(outs[0], base[0]) and torch.equal(outs[3], base[3])
    assert torch.equal(gout, gk)


# ------------------------------------------------------------------------------------------------
# fused front end: RolloutEngine.evaluate_knots (knots -> cost, grad_knots in one C call)
# ------------------------------------------------------------------------------------------------
def _smooth_knots(rm, B, nk, seed):
    """knots around a joint-space random walk, inside the joint limits"""
    from helpers import random_walk_q
    return random_walk_q(rm, B, nk, seed=seed).astype(np.float32)


@pytest.mark.parametrize("mode", ["trajopt_swept", "discrete"])
@pytest.mark.parametrize("degree,steps,implicit", [(4, 4, False), (3, 2, True), (5, 1, False)])
def test_fused_knots_rollout_vs_oracle_chain(mode, degree, steps, implicit):
    """evaluate_knots == oracle chain  bspline_forward -> rollout_cost_grad -> bspline_backward  and
    == our own unfused chain (spline kernel -> evaluate_action -> adjoint kernel) to float rounding
    (bit for bit whenever both run the same instantiation of the row code)."""
    from helpers import random_q, small_voxel_world
    from curobo_b200.robot_model import load_robot
    from curobo_b200.rollout import RolloutConfig, RolloutEngine
    from curobo_b200.scene import CuboidData, VoxelData
    from curobo_b200.world import make_benchmark_cuboid_world
    from oracle import rollout_oracle as O

    rm = load_robot("franka")
    B, nk, D = 4, 8, rm.num_dof
    Tn = bo.padded_horizon_for(nk, degree, steps)
    rng = np.random.default_rng(7)
    knots = _smooth_knots(rm, B, nk, seed=80 + degree)
    q0 = knots[:, 0] + rng.normal(0, 0.02, size=(B, D)).astype(np.float32)
    z = np.zeros((B, D), np.float32)
    start = (q0, rng.normal(0, 0.1, (B, D)).astype(np.float32), z, z)
    goal = (knots[:, -1].copy(), z, z, z)
    sidx = np.arange(B, dtype=np.int32)
    gidx = np.arange(B, dtype=np.int32)
    traj_dt = np.full(B, 0.05, np.float32)
    imp = np.full(B, int(implicit), np.uint8)

    cfg = RolloutConfig.trajopt()
    if mode == "discrete":
        cfg.use_sweep = False
        cfg.use_speed_metric = False
    cub, vox = make_benchmark_cuboid_world(), small_voxel_world()
    gq_ = random_q(rm, B, seed=61)
    _, _, gp, gqt = O.fk_forward(rm, gq_)
    gp, gqt = gp[:, :, None, :].copy(), gqt[:, :, None, :].copy()
    eng = RolloutEngine(rm, cfg, DEV, CuboidData.from_world(cub, DEV), VoxelData.from_world(vox, DEV))
    nt = torch.zeros((1, 6), dtype=torch.float32, device=DEV)
    eng.update_goal(T(gp), T(gqt), T(sidx), non_terminal_axes=nt)
    start_t = JointState(*[T(x) for x in start])
    goal_t = JointState(*[T(x) for x in goal], dt=T(traj_dt))
    out = eng.evaluate_knots(T(knots), start_t, T(sidx), goal_t, T(gidx), T(imp), bspline_degree=degree,
                             interpolation_steps=steps, store_state=True, in_kernel_spline=True)
    torch.cuda.synchronize()
    cost, gk = out.cost.clone(), out.grad_knots.clone()
    state = [t.clone() for t in eng._state]
    # the default (expanded, 3-launch) schedule of the same call gives the same bits
    out = eng.evaluate_knots(T(knots), start_t, T(sidx), goal_t, T(gidx), T(imp), bspline_degree=degree,
                             interpolation_steps=steps)
    torch.cuda.synchronize()
    # (different template instantiations of the row code: FMA contraction may differ in the last bit)
    torch.testing.assert_close(out.cost, cost, rtol=1e-5, atol=1e-6 * float(cost.abs().max()))
    torch.testing.assert_close(out.grad_knots, gk, rtol=1e-4, atol=1e-5 * float(gk.abs().max()))
    assert all(torch.equal(a, b) for a, b in zip(state, eng._state))

    # oracle chain
    p, v, a, j, odt = bo.bspline_forward(knots, start, goal, sidx, gidx, traj_dt, imp, Tn, degree)
    for g, w in zip(state, (p, v, a, j)):
        assert np.allclose(g.cpu().numpy(), w, rtol=2e-5, atol=2e-5 * max(1.0, np.abs(w).max()))
    ocfg = cfg.to_oracle_cfg(1)
    ocfg["pose_non_terminal_axes"] = np.zeros((1, 6), np.float32)
    # the rollout oracle is fed the states the GPU produced (already checked against the spline oracle above): the
    # swept-collision sample count is a discontinuous function of the waypoint distance, so 1e-7 differences in q
    # between the two spline evaluations could otherwise flip a sample on or off
    sp, sv, sa, sj = (t.cpu().numpy() for t in state)
    want = O.rollout_cost_grad(rm, sp, ocfg, world_cuboid=cub, world_voxel=vox, goal_pos=gp, goal_quat=gqt, idxs_goal=sidx,
                               vel=sv, acc=sa, jerk=sj, dt=odt)
    np.testing.assert_allclose(cost.cpu().numpy(), want["cost_bh"], rtol=5e-4, atol=2e-5 * want["cost_bh"].max())
    gs = want["cspace_grads"]
    want_gk = bo.bspline_backward(want["grad_q"], gs[1], gs[2], gs[3], traj_dt, gidx, imp, nk, degree)
    np.testing.assert_allclose(gk.cpu().numpy(), want_gk, rtol=5e-3, atol=5e-5 * np.abs(want_gk).max())

    # our own unfused chain, same kernels: must agree exactly
    fn = StateFromBSplineKnot(DEV, D, batch_size=B, n_knots=nk, interpolation_steps=steps, use_implicit_goal_state=implicit,
                              control_space={3: ControlSpace.BSPLINE_3, 4: ControlSpace.BSPLINE_4, 5: ControlSpace.BSPLINE_5}[degree])
    seq = fn.forward(start_t, T(knots), JointState.zeros((B, Tn, D), DEV), start_state_idx=T(sidx), goal_state=goal_t,
                     goal_state_idx=T(gidx), use_implicit_goal_state=T(imp))
    for g, w in zip(state, (seq.position, seq.velocity, seq.acceleration, seq.jerk)):
        assert torch.equal(g, w)
    eng2 = RolloutEngine(rm, cfg, DEV, CuboidData.from_world(cub, DEV), VoxelData.from_world(vox, DEV))
    eng2.update_goal(T(gp), T(gqt), T(sidx), non_terminal_axes=nt)
    o2 = eng2.evaluate_action(seq.position, vel=seq.velocity, acc=seq.acceleration, jerk=seq.jerk, dt=T(traj_dt))
    torch.testing.assert_close(o2.cost, cost, rtol=1e-5, atol=1e-6 * float(cost.abs().max()))
    gk2 = torch.zeros_like(gk)
    trajectory_cu.launch_bspline_interpolation_backward_kernel(gk2, o2.grad_q, o2.grad_vel, o2.grad_acc, o2.grad_jerk,
                                                               T(traj_dt), T(gidx), T(imp), B, Tn, D, nk, degree)
    torch.testing.assert_close(gk2, gk, rtol=1e-4, atol=1e-5 * float(gk.abs().max()))


def test_fused_knots_full_size_mpc_and_graph():
    """MPC scale: 1024 seeds x 16 knots (degree 4, 1 step -> 22 rows) on the 256^3 ESDF, swept + speed metric.
    Fused == unfused chain, and the call is CUDA-graph capturable."""
    from curobo_b200.robot_model import load_robot
    from curobo_b200.rollout import RolloutConfig, RolloutEngine
    from curobo_b200.scene import VoxelData
    from curobo_b200.world import make_box_esdf

    rm = load_robot("franka")
    B, nk, D, degree, steps = 1024, 16, rm.num_dof, 4, 1
    Tn = bo.padded_horizon_for(nk, degree, steps)
    sdf = make_box_esdf(n=256, voxel_size=0.01, num_boxes=12, seed=0, xp=torch)
    vox = VoxelData(T(np.array([[[256, 256, 256, 0.01]]], np.float32)), T(np.array([[[0, 0, 0, 1, 0, 0, 0, 0]]], np.float32)),
                    torch.ones((1, 1), dtype=torch.uint8, device=DEV), torch.ones(1, dtype=torch.int32, device=DEV),
                    sdf.reshape(1, 1, -1).contiguous(), 1, 1, 100.0)
    knots = T(_smooth_knots(rm, B, nk, seed=90))
    z = torch.zeros((1, D), device=DEV)
    start = JointState(knots[:1, 0].contiguous(), z, z, z)
    goal = JointState(knots[:1, -1].contiguous(), z, z, z, dt=torch.full((1,), 0.05, device=DEV))
    zi = torch.zeros(B, dtype=torch.int32, device=DEV)
    imp = torch.zeros(1, dtype=torch.uint8, device=DEV)
    cfg = RolloutConfig.trajopt()
    eng = RolloutEngine(rm, cfg, DEV, voxel=vox)
    out = eng.evaluate_knots(knots, start, zi, goal, zi, imp, degree, steps, in_kernel_spline=True)
    torch.cuda.synchronize()
    cost, gk = out.cost.clone(), out.grad_knots.clone()
    out = eng.evaluate_knots(knots, start, zi, goal, zi, imp, degree, steps)
    torch.cuda.synchronize()
    assert torch.equal(out.cost, cost) and torch.equal(out.grad_knots, gk)
    assert torch.isfinite(cost).all() and torch.isfinite(gk).all() and float(gk.abs().max()) > 0

    fn = StateFromBSplineKnot(DEV, D, batch_size=B, n_knots=nk, interpolation_steps=steps, control_space=ControlSpace.BSPLINE_4)
    seq = fn.forward(start, knots, JointState.zeros((B, Tn, D), DEV), start_state_idx=zi, goal_state=goal, goal_state_idx=zi,
                     use_implicit_goal_state=imp)
    eng2 = RolloutEngine(rm, cfg, DEV, voxel=vox)
    o2 = eng2.evaluate_action(seq.position, vel=seq.velocity, acc=seq.acceleration, jerk=seq.jerk,
                              dt=torch.full((B,), 0.05, device=DEV))
    assert torch.equal(o2.cost, cost)
    gk2 = torch.zeros_like(gk)
    trajectory_cu.launch_bspline_interpolation_backward_kernel(gk2, o2.grad_q, o2.grad_vel, o2.grad_acc, o2.grad_jerk, goal.dt,
                                                               zi, imp, B, Tn, D, nk, degree)
    assert torch.equal(gk2, gk)

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        eng.evaluate_knots(knots, start, zi, goal, zi, imp, degree, steps)   # warm the plan cache outside capture
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            eng.evaluate_knots(knots, start, zi, goal, zi, imp, degree, steps)
        eng.out.cost.zero_()
        eng.out.grad_knots.zero_()
        graph.replay()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    assert torch.equal(eng.out.cost, cost) and torch.equal(eng.out.grad_knots, gk)
