"""GPU parity of the RNEA inverse-dynamics kernels (SURVEY.md 8f rank 3) through the C ABI
(curobo_b200.backends.dynamics) against the numpy oracle and the REFERENCE's own kernels (outputs recorded on a B200,
tests/ref_kernels.py; serial threads_per_batch = 1 path: same order of every sum -> expected equal to float rounding, rtol 1e-5)."""
import numpy as np
import pytest
import torch

import ref_kernels
from dynamics_cases import CASES, make_case, model_args, pack_cache
from curobo_b200.backends import dynamics as dynamics_cu
from curobo_b200.dynamics import Dynamics
from oracle import dynamics_oracle as do

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def T(a, dt=None):
    t = torch.as_tensor(np.ascontiguousarray(a)).to(DEV)
    return t.to(dt) if dt is not None else t


def dev_model(c):
    m = model_args(c)
    return tuple(T(x) for x in m) + (T(c["starts"]), T(c["order"]))


def close(a, b, rtol, what=""):
    a, b = np.asarray(a), np.asarray(b)
    assert np.allclose(a, b, rtol=rtol, atol=rtol * max(float(np.abs(b).max()), 1e-30)), (what, float(np.abs(a - b).max()))


@pytest.mark.parametrize("robot,B,seed", CASES + [("franka", 1000, 4), ("g1_29", 300, 5)])
def test_rnea_vs_oracle_and_reference(robot, B, seed):
    c = make_case(robot, B, seed)
    model = dev_model(c)
    nl, D, nlev = c["nl"], c["D"], c["n_levels"]
    q, qd, qdd, gt = T(c["q"]), T(c["qd"]), T(c["qdd"]), T(c["grad_tau"])
    tau = torch.full((B, D), float("nan"), device=DEV)
    cache = torch.zeros((B, nl * 20), device=DEV)
    dynamics_cu.launch_rnea_forward(tau, q, qd, qdd, *model, cache, B, nl, D, nlev)
    gq, gqd, gqdd = (torch.full((B, D), float("nan"), device=DEV) for _ in range(3))
    dynamics_cu.launch_rnea_backward(gq, gqd, gqdd, gt, q, qd, *model, cache, B, nl, D, nlev)
    torch.cuda.synchronize()
    if B <= 16:
        m = model_args(c)
        tau_w, cache_w = do.rnea_forward(c["q"], c["qd"], c["qdd"], *m)
        close(tau.cpu().numpy(), tau_w, 1e-4, "tau vs oracle")
        close(cache.cpu().numpy().reshape(B, nl, 20)[:, :, :18], pack_cache(cache_w, nl).reshape(B, nl, 20)[:, :, :18], 1e-4, "cache")
        want = do.rnea_backward(c["grad_tau"], c["q"], c["qd"], cache_w, *m)
        for g, w, n in zip((gq, gqd, gqdd), want, ("grad_q", "grad_qd", "grad_qdd")):
            close(g.cpu().numpy(), w, 3e-4, n + " vs oracle")
    if ref_kernels.comparing():
        def reference():
            rt, rc = ref_kernels.rnea_forward(model, q, qd, qdd, nl, D, nlev)
            return [rt, rc] + ref_kernels.rnea_backward(model, gt, q, qd, rc, nl, D, nlev)
        r = ref_kernels.recorded(("dynamics", "rnea", robot, B, seed), reference)
        close(r.at(0, tau.cpu().numpy()), r[0], 1e-5, "tau vs reference")
        close(r.at(1, cache.cpu().numpy()).reshape(-1, nl, 20)[:, :, :18], r[1].reshape(-1, nl, 20)[:, :, :18], 1e-5,
              "cache vs reference")
        for i, (g, n) in enumerate(zip((gq, gqd, gqdd), ("grad_q", "grad_qd", "grad_qdd"))):
            close(r.at(2 + i, g.cpu().numpy()), r[2 + i], 2e-5, n + " vs reference")
        # caches are interchangeable: our adjoint on the reference's cache (its recorded rows, the same rows as grad_q's)
        ir = torch.as_tensor(r.rows(1), device=DEV)
        g2 = [torch.zeros((len(ir), D), device=DEV) for _ in range(3)]
        dynamics_cu.launch_rnea_backward(*g2, gt[ir].contiguous(), q[ir].contiguous(), qd[ir].contiguous(), *model,
                                         T(r[1]), len(ir), nl, D, nlev)
        close(g2[0].cpu().numpy(), r[2], 2e-5, "adjoint on the reference cache")


def test_dynamics_operator_autograd_and_graph():
    """Dynamics.compute_inverse_dynamics is differentiable ([batch, horizon, dof] in), deterministic, graph-capturable."""
    c = make_case("franka", 64 * 8, 7)
    dyn = Dynamics(c["rm"], c["mc"], c["inn"], gravity=(0.0, 0.0, -9.81), device=DEV)
    shape = (64, 8, c["D"])
    q = T(c["q"]).view(shape).clone().requires_grad_(True)
    qd = T(c["qd"]).view(shape).clone().requires_grad_(True)
    qdd = T(c["qdd"]).view(shape).clone().requires_grad_(True)
    tau = dyn.compute_inverse_dynamics(q, qd, qdd)
    w = T(c["grad_tau"]).view(shape)
    (tau * w).sum().backward()
    m = model_args(c)
    tau_w, cache_w = do.rnea_forward(c["q"], c["qd"], c["qdd"], *m)
    close(tau.detach().cpu().numpy().reshape(-1, c["D"]), tau_w, 1e-4)
    want = do.rnea_backward(c["grad_tau"], c["q"], c["qd"], cache_w, *m)
    for g, wv in zip((q.grad, qd.grad, qdd.grad), want):
        close(g.cpu().numpy().reshape(-1, c["D"]), wv, 3e-4)
    t1 = dyn.compute_inverse_dynamics(q.detach(), qd.detach(), qdd.detach()).clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            t2 = dyn.compute_inverse_dynamics(q.detach(), qd.detach(), qdd.detach())
        dyn._tau.zero_()
        graph.replay()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    assert torch.equal(t1, t2)
    with pytest.raises(ValueError):
        Dynamics(c["rm"], c["mc"], c["inn"], device="cpu")


@pytest.mark.parametrize("robot,B", [("franka", 2), ("g1_29", 37)])
def test_rnea_external_wrenches(robot, B):
    """f_ext enters f = I a + v x* I v - f_ext (rnea_forward_kernel.cuh:206-216); tau is linear in it, so grad_f_ext of
    <grad_tau, tau> is checked exactly (to rounding) by differencing the oracle along a few wrench components."""
    c = make_case(robot, B, 11)
    model = dev_model(c)
    m = model_args(c)
    nl, D, nlev = c["nl"], c["D"], c["n_levels"]
    rng = np.random.default_rng(5)
    fe = rng.normal(size=(B, nl, 6)).astype(np.float32) * 3.0
    q, qd, qdd, gt = T(c["q"]), T(c["qd"]), T(c["qdd"]), T(c["grad_tau"])
    tau = torch.zeros((B, D), device=DEV)
    cache = torch.zeros((B, nl * 20), device=DEV)
    dynamics_cu.launch_rnea_forward(tau, q, qd, qdd, *model, cache, B, nl, D, nlev, f_ext=T(fe))
    tau_w, cache_w = do.rnea_forward(c["q"], c["qd"], c["qdd"], *m, f_ext=fe)
    close(tau.cpu().numpy(), tau_w, 1e-4, "tau with f_ext")
    g = [torch.zeros((B, D), device=DEV) for _ in range(3)]
    gfe = torch.full((B, nl, 6), float("nan"), device=DEV)
    dynamics_cu.launch_rnea_backward(*g, gt, q, qd, *model, cache, B, nl, D, nlev, grad_f_ext=gfe)
    want = do.rnea_backward(c["grad_tau"], c["q"], c["qd"], cache_w, *m)
    for got, w in zip(g, want):
        close(got.cpu().numpy(), w, 3e-4, "grads with f_ext")
    got = gfe.cpu().numpy()
    assert np.isfinite(got).all()
    tau0 = do.rnea_forward(c["q"], c["qd"], c["qdd"], *m)[0].astype(np.float64)
    for k, i in [(nl - 1, 0), (nl - 1, 4), (nl // 2, 2), (1, 5), (0, 3)]:
        e = np.zeros((B, nl, 6), np.float32)
        e[:, k, i] = 1.0
        dt = do.rnea_forward(c["q"], c["qd"], c["qdd"], *m, f_ext=e)[0].astype(np.float64) - tau0
        w = (c["grad_tau"].astype(np.float64) * dt).sum(-1)
        assert np.allclose(got[:, k, i], w, rtol=2e-3, atol=2e-3 * max(1.0, np.abs(w).max())), (k, i, got[:, k, i], w)


def test_rnea_row_kernels_match_cta_kernels(monkeypatch):
    """CB200_RNEA_ROWS=1 selects the thread-per-row kernels (the path for trees too large for the CTA tile)."""
    c = make_case("g1_29", 77, 13)
    model = dev_model(c)
    nl, D, nlev, B = c["nl"], c["D"], c["n_levels"], 77
    q, qd, qdd, gt = T(c["q"]), T(c["qd"]), T(c["qdd"]), T(c["grad_tau"])
    outs = []
    for rows in (False, True):
        if rows:
            monkeypatch.setenv("CB200_RNEA_ROWS", "1")
        tau = torch.zeros((B, D), device=DEV)
        cache = torch.zeros((B, nl * 20), device=DEV)
        dynamics_cu.launch_rnea_forward(tau, q, qd, qdd, *model, cache, B, nl, D, nlev)
        g = [torch.zeros((B, D), device=DEV) for _ in range(3)]
        dynamics_cu.launch_rnea_backward(*g, gt, q, qd, *model, cache, B, nl, D, nlev)
        torch.cuda.synchronize()
        outs.append([tau.cpu().numpy(), cache.cpu().numpy()] + [x.cpu().numpy() for x in g])
    for a_, b_ in zip(*outs):
        close(a_, b_, 2e-5, "row kernels vs CTA kernels")
