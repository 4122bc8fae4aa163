"""GPU parity of the optimizer-side kernels (SURVEY.md 8f rank 2) through the C ABI
(curobo_b200.backends.optimization) against the numpy oracle and the REFERENCE's own kernels (their outputs recorded on a
B200, tests/ref_kernels.py), and the whole loop (L-BFGS step -> fused rollout -> line search) solving real problems.

Sums are associated like the reference's block reductions, so float results are expected bit-equal to the reference
kernels; the tests assert rtol 1e-6 and report exact equality where it must hold (copies, indices, counters).
"""
import numpy as np
import pytest
import torch

import ref_kernels
from optim_cases import LBFGS_CASES, LS_CASES, lbfgs_case, lbfgs_id, line_search_case, ls_id
from curobo_b200.backends import optimization as optimization_cu
from curobo_b200.optim import LBFGScu, LBFGSOpt, LBFGSOptCfg
from oracle import optim_oracle as oo

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def T(a, dt=None):
    t = torch.as_tensor(np.ascontiguousarray(a)).to(DEV)
    return t.to(dt) if dt is not None else t


def close(a, b, rtol=1e-6):
    a, b = np.asarray(a), np.asarray(b)
    assert np.allclose(a, b, rtol=rtol, atol=rtol * max(float(np.abs(b).max()), 1e-30)), float(np.abs(a - b).max())


def run_ours_lbfgs(c, **kw):
    t = {k: T(v) for k, v in c.items()}
    m, B, V = c["Y"].shape
    step = torch.full((B, V), float("nan"), device=DEV)
    optimization_cu.launch_lbfgs_step(step, t["rho"], t["Y"], t["S"], t["q"], t["grad_q"], t["x_0"], t["grad_0"], 0.01, B, m, V,
                                      True, True, **kw)
    return step, t


@pytest.mark.parametrize("kw", LBFGS_CASES, ids=lbfgs_id)
def test_lbfgs_step_vs_oracle_and_reference(kw):
    c = lbfgs_case(**kw)
    step, t = run_ours_lbfgs(c)
    w_step, w_rho, w_Y, w_S, w_x0, w_g0 = oo.lbfgs_step(c["rho"], c["Y"], c["S"], c["q"], c["grad_q"], c["x_0"], c["grad_0"],
                                                        0.01, True)
    assert np.array_equal(t["Y"].cpu().numpy(), w_Y) and np.array_equal(t["S"].cpu().numpy(), w_S)
    assert np.array_equal(t["x_0"].cpu().numpy(), w_x0) and np.array_equal(t["grad_0"].cpu().numpy(), w_g0)
    close(t["rho"].cpu().numpy(), w_rho, 2e-6)
    close(step.cpu().numpy(), w_step, 1e-4)       # oracle divides exactly, the kernel with --prec-div=false
    V, m = kw["V"], kw["m"]
    fits_shared = (((2 * V) + 2) * m + 32 + 1) * 4 <= 65536      # optimization_config.py:96-117
    # The reference has two variants.  The shared-memory one is what LBFGSOpt uses whenever the history fits 64 KB
    # (lbfgs.py:171-184, lbfgs_ik.yml / lbfgs_bspline_trajopt.yml: use_cuda_kernel_shared_buffers true) and is the
    # parity target.  Its global-memory fallback disagrees with it by 10-50 % and is not even run-to-run deterministic
    # for v_dim > 32 (measured on B200: scripts/debug_lbfgs.py), so it is only compared for single-warp problems.
    variants = ([True] if fits_shared else []) + ([False] if V <= 32 else [])
    if ref_kernels.comparing() and m in (3, 5, 7, 15, 27, 31):
        ours = [a.cpu().numpy() for a in (step, t["rho"], t["Y"], t["S"], t["x_0"])]

        def reference(shared):
            r = {k: T(v) for k, v in c.items()}
            rstep = torch.zeros_like(step)
            ref_kernels.lbfgs_step(rstep, r["rho"], r["Y"], r["S"], r["q"], r["x_0"], r["grad_0"], r["grad_q"], 0.01, True, shared)
            return rstep, r["rho"], r["Y"], r["S"], r["x_0"]
        for shared in variants:
            ref = ref_kernels.recorded(("optim", "lbfgs_step", lbfgs_id(kw), shared), lambda: reference(shared))
            o_step, o_rho, o_Y, o_S, o_x0 = (ref.at(i, a) for i, a in enumerate(ours))
            assert np.array_equal(o_Y, ref[2]) and np.array_equal(o_S, ref[3]) and np.array_equal(o_x0, ref[4])
            close(o_rho, ref[1], 1e-6)
            close(o_step, ref[0], 1e-6)


def test_lbfgs_autograd_function_and_search_points():
    """LBFGScu.apply (reference buffer shapes [m,B,V,1]) and the fused line-search set-up extension."""
    c = lbfgs_case(seed=21, B=19, V=7, m=7)
    t = {k: T(v) for k, v in c.items()}
    m, B, V = c["Y"].shape
    step_buf = torch.zeros((B, V), device=DEV)
    dq = LBFGScu.apply(step_buf, t["rho"].view(m, B, 1, 1), t["Y"].view(m, B, V, 1), t["S"].view(m, B, V, 1), t["q"],
                       t["grad_q"].view(B, 1, V), t["x_0"].view(B, V, 1), t["grad_0"].view(B, V, 1), 0.01, True, True)
    want = oo.lbfgs_step(c["rho"], c["Y"], c["S"], c["q"], c["grad_q"], c["x_0"], c["grad_0"], 0.01, True)[0]
    close(dq.cpu().numpy(), want, 1e-4)
    # fused search points: x_set = q + mags * scale_action(step)
    mags = T(np.array([0.0, 0.1, 0.5, 1.0], np.float32))
    step_max = T((np.abs(want).max(0) * 0.5).astype(np.float32))      # forces clamping for some problems
    x_set = torch.zeros((B, 4, V), device=DEV)
    scaled = torch.zeros((B, V), device=DEV)
    step, _ = run_ours_lbfgs(c, x_set=x_set, step_scaled=scaled, search_magnitudes=mags, action_step_max=step_max)
    s_np = step.cpu().numpy()
    ratio = np.maximum((np.abs(s_np) / step_max.cpu().numpy()[None]).max(1), 1.0)
    assert (ratio > 1).any() and (ratio == 1).any()
    close(scaled.cpu().numpy(), s_np / ratio[:, None], 1e-5)
    close(x_set.cpu().numpy(), c["q"][:, None, :] + mags.cpu().numpy()[None, :, None] * scaled.cpu().numpy()[:, None, :], 1e-6)
    with pytest.raises(RuntimeError, match="History_m greater than 31"):
        optimization_cu.launch_lbfgs_step(step, t["rho"], t["Y"], t["S"], t["q"], t["grad_q"], t["x_0"], t["grad_0"], 0.01, B, 32,
                                          V, True, True)


def ls_state(c, B, n, V):
    z = lambda *s, dt=torch.float32: torch.zeros(s, device=DEV, dtype=dt)  # noqa: E731
    return dict(best_cost=T(c["best_cost"]), best_action=T(c["best_action"]), best_iteration=T(c["best_iteration"]),
                current_iteration=T(c["current_iteration"]), converged=z(B, dt=torch.uint8), exploration_cost=z(B),
                exploration_action=z(B, V), exploration_gradient=z(B, V), exploration_idx=z(B * n, dt=torch.int32),
                selected_cost=z(B), selected_action=z(B, V), selected_gradient=z(B, V), selected_idx=z(B * n, dt=torch.int32))


@pytest.mark.parametrize("kw", LS_CASES, ids=ls_id)
@pytest.mark.parametrize("strong,approx", [(False, True), (False, False), (True, False)])
def test_line_search_vs_oracle_and_reference(kw, strong, approx):
    c = line_search_case(**kw)
    B, n, V = c["search_action"].shape
    st = ls_state(c, B, n, V)
    sc, sa, sg, sd, mg = T(c["search_cost"]), T(c["search_action"]), T(c["search_gradient"]), T(c["step_direction"]), T(c["magnitudes"])
    optimization_cu.launch_line_search(
        st["best_cost"], st["best_action"], st["best_iteration"], st["current_iteration"], st["converged"], 10, 0.0, 0.0,
        st["exploration_cost"], st["exploration_action"], st["exploration_gradient"], st["exploration_idx"], st["selected_cost"],
        st["selected_action"], st["selected_gradient"], st["selected_idx"], sc, sa, sg, sd, mg, 1e-5, 0.9, strong, approx, n, V, B)
    o = oo.line_search(c["best_cost"], c["best_action"], c["best_iteration"], c["current_iteration"], 10, 0.0, 0.0,
                       c["search_cost"], c["search_action"], c["search_gradient"], c["step_direction"], c["magnitudes"], 1e-5, 0.9,
                       strong, approx)
    got = {k: v.cpu().numpy() for k, v in st.items()}
    # a directional derivative within float rounding of a threshold may legitimately flip between orders of summation;
    # the oracle reproduces the kernel's order, so every output is compared exactly
    assert np.array_equal(got["selected_idx"].reshape(B, n), o["selected_idx"])
    assert np.array_equal(got["exploration_idx"].reshape(B, n), o["exploration_idx"])
    for k in ("selected_cost", "selected_action", "selected_gradient", "exploration_cost", "exploration_action",
              "exploration_gradient", "best_cost", "best_action", "best_iteration", "current_iteration", "converged"):
        assert np.array_equal(got[k], o[k]), k
    if ref_kernels.comparing() and V >= n:      # the reference kernel needs opt_dim >= n_linesearch threads
        def reference():
            rs = ref_kernels.line_search(ls_state(c, B, n, V), sc, sa, sg, sd, mg, 1e-5, 0.9, strong, approx)
            return [rs[k] for k in st]
        ref = ref_kernels.recorded(("optim", "line_search", ls_id(kw), strong, approx), reference)
        for i, k in enumerate(st):
            assert np.array_equal(ref.at(i, got[k]), ref[i]), k


def test_lbfgs_opt_solves_quadratics():
    """The whole loop on batched convex quadratics (cost/grad in torch): every problem reaches its minimiser."""
    torch.manual_seed(0)
    B, V = 64, 7
    A = torch.randn(B, V, V, device=DEV)
    A = A @ A.transpose(1, 2) + 0.5 * torch.eye(V, device=DEV)
    bvec = torch.randn(B, V, device=DEV)
    n = 4

    def cost_grad(x):                      # x [B*n, V]
        xb = x.view(B, n, V)
        Ax = torch.einsum("bij,bnj->bni", A, xb)
        c = 0.5 * (xb * Ax).sum(-1) - (bvec[:, None, :] * xb).sum(-1) + 30.0      # keep costs positive (relative test)
        return c.reshape(-1).contiguous(), (Ax - bvec[:, None, :]).reshape(B * n, V).contiguous()

    lows, highs = torch.full((V,), -10.0, device=DEV), torch.full((V,), 10.0, device=DEV)
    opt = LBFGSOpt(LBFGSOptCfg(num_iters=60, initial_step_scale=0.01), B, 1, V, lows, highs, cost_grad, DEV)
    x = opt.optimize(torch.randn(B, V, device=DEV)).view(B, V)
    x_star = torch.linalg.solve(A, bvec)
    # fp32 Armijo tests on costs of magnitude ~30 stop resolving improvements below ~1e-5 relative
    assert float((x - x_star).abs().max()) < 1e-2
    c_star = (0.5 * (x_star * torch.einsum("bij,bj->bi", A, x_star)).sum(-1) - (bvec * x_star).sum(-1) + 30.0)
    assert float(((opt.best_cost - c_star) / c_star).abs().max()) < 1e-5
    assert int(opt.current_iteration.min()) == 60
    assert torch.isfinite(opt.best_cost).all()


def test_ik_solve_end_to_end():
    """512-goal-style IK at small scale through the public pieces: LBFGSOpt driving RolloutEngine.evaluate_action on
    [problems x seeds x 4 line-search candidates] rows, 3 launches per iteration.  Reachable goals (FK of random
    configurations), 16 seeds each: at least 90 % of the goals end with a seed below 5 mm / 0.05 rad-ish pose error."""
    from helpers import random_q
    from curobo_b200.kinematics import Kinematics
    from curobo_b200.robot_model import load_robot
    from curobo_b200.rollout import RolloutConfig, RolloutEngine
    from oracle import rollout_oracle as O

    rm = load_robot("franka")
    P, seeds, n = 24, 16, 4
    B = P * seeds
    D = rm.num_dof
    q_goal = random_q(rm, P, seed=5) * 0.7
    _, _, gp, gq = O.fk_forward(rm, q_goal)
    cfg = RolloutConfig.ik()
    cfg.self_weight = 0.0     # pose + joint limits only: unobstructed IK
    cfg.scene_weight = 0.0
    eng = RolloutEngine(rm, cfg, DEV)
    idx = torch.arange(B, device=DEV, dtype=torch.int32).div(seeds, rounding_mode="floor").repeat_interleave(n).to(torch.int32)
    eng.update_goal(T(gp[:, :, None, :]), T(gq[:, :, None, :]), idx.contiguous())

    def cost_grad(x):
        out = eng.evaluate_action(x.view(B * n, 1, D))
        return out.cost.view(-1), out.grad_q.view(B * n, D)

    lows, highs = T(rm.position_limits[0]), T(rm.position_limits[1])
    opt = LBFGSOpt(LBFGSOptCfg(num_iters=100), B, 1, D, lows, highs, cost_grad, DEV)
    x0 = T(random_q(rm, B, seed=6))
    q_sol = opt.optimize(x0).view(B, D)
    torch.cuda.synchronize()
    assert torch.isfinite(q_sol).all()
    st = Kinematics(rm, DEV).compute_kinematics(q_sol.view(B, 1, D))
    pos = st.tool_pose_position.reshape(B, -1, 3)[:, 0].detach().cpu().numpy().reshape(P, seeds, 3)
    err = np.linalg.norm(pos - gp[:, 0][:, None, :], axis=-1)       # [P, seeds]
    solved = (err.min(axis=1) < 5e-3)
    assert solved.mean() >= 0.9, (solved.mean(), np.sort(err.min(axis=1))[-5:])
    assert float(opt.best_cost.view(P, seeds).min(dim=1)[0].max()) < float(opt.best_cost.max()) + 1e-6
