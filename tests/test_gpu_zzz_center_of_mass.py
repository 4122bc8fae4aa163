"""Centre of mass of the FK operator (`compute_com`, SURVEY.md 8a rows a2 / a4: `com[B,H,4]` is one of the outputs of
launch_kinematics_forward_spheres, its gradient one of the inputs of launch_kinematics_backward): kin_forward_kernel<true> /
kin_backward_kernel<true> against numpy (mass-weighted mean of the links' world centres of mass from the oracle's cumulative
transforms) and finite differences.  Written after round 1's GPU budget was spent: passes on the emulated kernels, has not run on a
B200 yet, ordered late."""
import numpy as np
import pytest
import torch

from helpers import humanoid_q, random_q
from curobo_b200.kinematics import Kinematics
from curobo_b200.robot_model import load_robot
from oracle import rollout_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def T(a):
    return torch.as_tensor(np.ascontiguousarray(a)).to(DEV)


def com_numpy(rm, q):
    cum = O.fk_forward(rm, q)[0].astype(np.float64).reshape(q.shape[0], rm.num_links, 3, 4)
    mc = np.asarray(rm.link_masses_com, np.float64)
    w = np.where(mc[:, 3] > 0, mc[:, 3], 0.0)
    world = np.einsum("blij,lj->bli", cum[..., :3], mc[:, :3]) + cum[..., 3]
    M = w.sum()
    return (world * w[None, :, None]).sum(1) / M, M


@pytest.mark.parametrize("robot,n", [("franka", 33), ("g1_29", 9)])
def test_center_of_mass_and_its_gradient(robot, n):
    import dataclasses
    rm = load_robot(robot)
    rng = np.random.default_rng(4)
    mc = np.zeros((rm.num_links, 4), np.float32)
    mc[:, :3] = rng.uniform(-0.05, 0.05, (rm.num_links, 3))
    mc[:, 3] = rng.uniform(0.2, 3.0, rm.num_links)
    mc[rm.num_links // 2, 3] = 0.0                        # a massless link is skipped
    rm = dataclasses.replace(rm, link_masses_com=mc)
    q = (random_q(rm, n, seed=6) if robot == "franka" else humanoid_q(rm, n, seed=6)).astype(np.float32)
    kin = Kinematics(rm, DEV, compute_com=True)
    qt = T(q).requires_grad_(True)
    st = kin.compute_kinematics(qt)
    want, M = com_numpy(rm, q)
    got = st.center_of_mass.detach().cpu().numpy().reshape(n, 4)
    assert np.allclose(got[:, :3], want, atol=2e-5) and np.allclose(got[:, 3], M, rtol=1e-6)
    g = rng.normal(size=(n, 4)).astype(np.float32)
    gs = rng.normal(size=tuple(st.robot_spheres.shape)).astype(np.float32) * 0.1
    ((st.center_of_mass.view(n, 4) * T(g)).sum() + (st.robot_spheres * T(gs)).sum()).backward()
    got_g = qt.grad.cpu().numpy()
    # reference gradient: spheres part from the FK-backward oracle, CoM part by central differences of the numpy CoM
    cum, sph, pos, quat = O.fk_forward(rm, q)
    base = O.fk_backward(rm, cum, gs.reshape(sph.shape), np.zeros_like(pos), np.zeros_like(quat))
    fd = np.zeros_like(base, dtype=np.float64)
    eps = 1e-3
    for d in range(rm.num_dof):
        qp, qm = q.astype(np.float64).copy(), q.astype(np.float64).copy()
        qp[:, d] += eps
        qm[:, d] -= eps
        cp, cm = com_numpy(rm, qp.astype(np.float32))[0], com_numpy(rm, qm.astype(np.float32))[0]
        fd[:, d] = ((cp - cm) / (2 * eps) * g[:, :3]).sum(-1)
    want_g = base + fd
    assert np.allclose(got_g, want_g, rtol=5e-3, atol=5e-3 * np.abs(want_g).max()), float(np.abs(got_g - want_g).max())
    # without compute_com the operator is what it was
    st0 = Kinematics(rm, DEV).compute_kinematics(T(q))
    assert st0.center_of_mass is None and torch.equal(st0.robot_spheres, st.robot_spheres.detach())
    import ref_kernels
    if ref_kernels.comparing():      # the reference's own kernels, COMPUTE_COM = true (launcher never run on a GPU yet: soft)
        def reference():
            rs, rc, rcom = ref_kernels.fk_forward_com(kin.params, T(q))
            zp = torch.zeros((n, rm.num_tool_frames, 3), device=DEV)
            zq = torch.zeros((n, rm.num_tool_frames, 4), device=DEV)
            return rcom, ref_kernels.fk_backward_com(kin.params, rc, rcom, zp, zq, T(gs).view(n, -1, 4).contiguous(), T(g))
        r = ref_kernels.recorded(("com", "fk_com", robot, n), reference)
        ok = np.allclose(r.at(0, got), r[0], rtol=1e-5, atol=2e-6) and \
            np.allclose(r.at(1, got_g), r[1], rtol=2e-3, atol=2e-5 * np.abs(r[1]).max())
        if not ok:
            pytest.xfail("differs from the reference's COMPUTE_COM kernels (reference launcher unvalidated on a GPU)")
