"""GPU parity of every per-op kernel (called through the C ABI) against the oracle, the committed
golden fixtures and -- for FK / FK-backward / self-collision -- the REFERENCE's own CUDA kernels.

Stated tolerances (fp32, both sides compiled with --ftz --prec-div=false --prec-sqrt=false, different
reduction orders), SURVEY.md 8c:
  FK positions / spheres  abs 1e-5 m        quaternions  abs 1e-5 (up to sign)
  costs                   rel 1e-4 + abs 1e-6 * max
  gradients               rel 1e-3 + abs 1e-5 * |g|_inf
  self-collision worst pair index: exact (except exact fp ties)
"""
import os

import numpy as np
import pytest
import torch

import ref_kernels
from helpers import random_q, random_walk_q, small_voxel_world
from curobo_b200 import cost as cb_cost
from curobo_b200.kinematics import Kinematics, KinematicsParams, SelfCollisionCost
from curobo_b200.robot_model import load_robot
from curobo_b200.scene import (CollisionBuffer, CuboidData, SceneData, SphereObstacleCollision,
                               SweptSphereObstacleCollision, VoxelData)
from curobo_b200.world import CuboidWorld, make_benchmark_cuboid_world
from oracle import rollout_oracle as O
from voxel_cases import cases

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def T(a, dt=None):
    t = torch.as_tensor(np.ascontiguousarray(a)).to(DEV)
    return t.to(dt) if dt is not None else t


def quat_close(a, b, atol):
    d = np.minimum(np.abs(a - b).max(-1), np.abs(a + b).max(-1))
    assert d.max() <= atol, d.max()


def grad_close(a, b, rtol=1e-3, scale=1e-5):
    np.testing.assert_allclose(a, b, rtol=rtol, atol=scale * max(np.abs(b).max(), 1e-6))


# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("robot,n", [("franka", 64), ("franka", 1000), ("g1_29", 96), ("g1_43", 40)])
def test_fk_forward_vs_oracle_and_reference(robot, n):
    rm = load_robot(robot)
    q = random_q(rm, n, seed=21)
    kin = Kinematics(rm, DEV)
    st = kin.compute_kinematics(T(q))
    cum, sph, pos, quat = O.fk_forward(rm, q)
    np.testing.assert_allclose(st.cumul_mat.cpu().numpy().reshape(cum.shape), cum, atol=1e-5)
    np.testing.assert_allclose(st.robot_spheres.cpu().numpy().reshape(sph.shape), sph, atol=1e-5)
    np.testing.assert_allclose(st.tool_pose_position.cpu().numpy().reshape(pos.shape), pos, atol=1e-5)
    quat_close(st.tool_pose_quaternion.cpu().numpy().reshape(quat.shape), quat, 1e-5)
    assert (st.tool_pose_quaternion[..., 0] >= 0).all()
    if ref_kernels.comparing():
        r = ref_kernels.recorded(("parity", "fk_forward", robot, n), lambda: ref_kernels.fk_forward(kin.params, T(q)))
        # our kernel vs the reference kernel, and (pinning the oracle) oracle vs the reference kernel
        np.testing.assert_allclose(r.at(3, st.cumul_mat.cpu().numpy().reshape(cum.shape)), r[3], atol=1e-5)
        np.testing.assert_allclose(r.at(2, st.robot_spheres.cpu().numpy().reshape(sph.shape)), r[2], atol=1e-5)
        np.testing.assert_allclose(r[3], r.at(3, cum), atol=1e-5)
        np.testing.assert_allclose(r[2], r.at(2, sph), atol=1e-5)
        np.testing.assert_allclose(r[0], r.at(0, pos), atol=1e-5)
        quat_close(r[1], r.at(1, quat), 1e-5)


def test_fk_without_spheres_entry_point():
    """launch_kinematics_forward (the no-sphere entry of the backend module) == the sphere variant's poses."""
    from curobo_b200.backends import kinematics as kin_cu
    rm = load_robot("franka")
    kp = KinematicsParams.from_robot_model(rm, DEV)
    q = T(random_q(rm, 50, seed=4))
    st = Kinematics(rm, DEV).compute_kinematics(q.view(50, 1, -1))
    pos = torch.zeros((50, 1, kp.num_pose_links, 3), device=DEV)
    quat = torch.zeros((50, 1, kp.num_pose_links, 4), device=DEV)
    cum = torch.zeros((50, 1, kp.num_links, 3, 4), device=DEV)
    kin_cu.launch_kinematics_forward(pos, quat, None, cum, q, kp.fixed_transforms, None, kp.joint_map_type, kp.joint_map,
                                     kp.link_map, kp.tool_frame_map, kp.joint_offset_map, 50, 1, kp.num_dof)
    assert torch.equal(pos, st.tool_pose_position.detach()) and torch.equal(quat, st.tool_pose_quaternion.detach())
    with pytest.raises(ValueError, match="outside the hot-path scope"):
        kin_cu.launch_kinematics_forward_spheres_jacobian()


def test_fk_golden_vector_on_gpu():
    rm = load_robot("franka")
    kin = Kinematics(rm, DEV)
    st = kin.compute_kinematics(T(np.array([[0.0, -1.2, 0.0, -2.0, 0.0, 1.0, 0.0]], np.float32)))
    np.testing.assert_allclose(st.tool_pose_position.cpu().numpy().reshape(3), [6.0860e-02, -4.7547e-12, 7.6373e-01], atol=1e-5)
    np.testing.assert_allclose(st.tool_pose_quaternion.cpu().numpy().reshape(4), [0.0382, 0.9193, 0.3808, 0.0922], atol=1e-4)


def test_fk_forward_golden_fixture():
    g = np.load(os.path.join(GOLD, "franka_fk_self_b64.npz"))
    rm = load_robot("franka")
    st = Kinematics(rm, DEV).compute_kinematics(T(g["q"]))
    np.testing.assert_allclose(st.robot_spheres.cpu().numpy().reshape(g["spheres"].shape), g["spheres"], atol=1e-5)
    np.testing.assert_allclose(st.cumul_mat.cpu().numpy().reshape(g["cumul"].shape), g["cumul"], atol=1e-5)


def test_fk_multi_sphere_configs():
    """num_envs > 1: row n uses sphere set env_query_idx[n // horizon] (kinematics_forward_helper.cuh:232-233)."""
    rm = load_robot("franka")
    ls = np.stack([rm.link_spheres, rm.link_spheres * np.array([1, 1, 1, 0.5], np.float32)])
    rm2 = load_robot("franka")
    rm2.link_spheres = ls
    kin = Kinematics(rm2, DEV)
    q = random_walk_q(rm, 6, 3, seed=4)
    eq = np.array([0, 1, 1, 0, 1, 0], np.int32)
    st = kin.compute_kinematics(T(q), env_query_idx=T(eq))
    _, sph, _, _ = O.fk_forward(rm2, q.reshape(-1, 7), env_query_idx=eq, horizon=3)
    np.testing.assert_allclose(st.robot_spheres.cpu().numpy().reshape(sph.shape), sph, atol=1e-5)


@pytest.mark.parametrize("robot,n", [("franka", 200), ("g1_29", 64), ("g1_43", 24)])
@pytest.mark.parametrize("sparse", [False, True])
def test_fk_backward_vs_oracle_and_reference(robot, n, sparse):
    rm = load_robot(robot)
    rng = np.random.default_rng(5)
    q = random_q(rm, n, seed=22)
    cum, sph, pos, quat = O.fk_forward(rm, q)
    gs = rng.normal(size=sph.shape).astype(np.float32)
    if sparse:
        gs *= (rng.uniform(size=sph.shape[:2]) < 0.05)[..., None]
    gp = rng.normal(size=pos.shape).astype(np.float32)
    gq = rng.normal(size=quat.shape).astype(np.float32)
    want = O.fk_backward(rm, cum, gs, gp, gq)
    kin = Kinematics(rm, DEV)
    qt = T(q).requires_grad_(True)
    st = kin.compute_kinematics(qt)
    loss = (st.robot_spheres.view(sph.shape) * T(gs)).sum() + (st.tool_pose_position.view(pos.shape) * T(gp)).sum() \
        + (st.tool_pose_quaternion.view(quat.shape) * T(gq)).sum()
    loss.backward()
    got = qt.grad.cpu().numpy()
    grad_close(got, want)
    if ref_kernels.comparing():
        r = ref_kernels.recorded(("parity", "fk_backward", robot, n, sparse),
                                 lambda: ref_kernels.fk_backward(kin.params, T(cum), T(gp), T(gq), T(gs)))
        grad_close(r.at(0, got), r[0])
        grad_close(r.at(0, want), r[0])          # pins the oracle's backward


def test_fk_backward_mimic_and_negative_axis():
    """Mimic joints share a joint index; a -1 axis flips joint_offset.x (parser_urdf.py:283-300):
    synthetic 4-link chain exercising both, checked against oracle finite differences."""
    from curobo_b200.robot_model import RobotModel
    fx = np.zeros((4, 3, 4), np.float32)
    fx[:, :, :3] = np.eye(3)
    fx[1, :, 3], fx[2, :, 3], fx[3, :, 3] = [0.2, 0, 0], [0, 0.3, 0], [0, 0, 0.1]
    rm = RobotModel(
        name="toy", link_names=list("abcd"), joint_names=["j0", "j1"], tool_frames=["d"], fixed_transforms=fx,
        link_map=np.array([0, 0, 1, 2], np.int16), joint_map=np.array([-1, 0, 1, 0], np.int16),
        joint_map_type=np.array([-1, 5, 0, 3], np.int8),
        joint_offset_map=np.array([[1, 0], [-1, 0.1], [1, 0], [0.5, -0.2]], np.float32),
        tool_frame_map=np.array([3], np.int16),
        link_spheres=np.array([[0.1, 0, 0, 0.05], [0, 0.1, 0.1, 0.04], [0.05, 0.05, 0, 0.03]], np.float32),
        link_sphere_idx_map=np.array([1, 3, 3], np.int16), link_chain_data=np.array([0, 0, 1, 0, 1, 2, 0, 1, 2, 3], np.int16),
        link_chain_offsets=np.array([0, 1, 3, 6, 10], np.int16), joint_links_data=np.array([1, 3, 2], np.int16),
        joint_links_offsets=np.array([0, 2, 3], np.int16), joint_affects_endeffector=np.ones(2, bool),
        link_masses_com=np.zeros((4, 4), np.float32), collision_pairs=np.array([[0, 1], [0, 2]], np.int16),
        sphere_padding=np.zeros(3, np.float32), position_limits=np.array([[-2, -1], [2, 1]], np.float32),
        velocity_limits=np.ones((2, 2), np.float32), acceleration_limits=np.ones((2, 2), np.float32),
        jerk_limits=np.ones((2, 2), np.float32), effort_limits=np.ones((2, 2), np.float32),
        default_joint_position=np.zeros(2, np.float32))
    rng = np.random.default_rng(0)
    q = rng.uniform(-1, 1, size=(16, 2)).astype(np.float32)
    cum, sph, pos, quat = O.fk_forward(rm, q)
    gs = rng.normal(size=sph.shape).astype(np.float32)
    gp = rng.normal(size=pos.shape).astype(np.float32)
    gq = rng.normal(size=quat.shape).astype(np.float32)
    kin = Kinematics(rm, DEV)
    qt = T(q).requires_grad_(True)
    st = kin.compute_kinematics(qt)
    np.testing.assert_allclose(st.robot_spheres.detach().cpu().numpy().reshape(sph.shape), sph, atol=1e-6)
    ((st.robot_spheres.view(sph.shape) * T(gs)).sum() + (st.tool_pose_position.view(pos.shape) * T(gp)).sum()
     + (st.tool_pose_quaternion.view(quat.shape) * T(gq)).sum()).backward()
    grad_close(qt.grad.cpu().numpy(), O.fk_backward(rm, cum, gs, gp, gq))


# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("robot,n", [("franka", 256), ("g1_29", 48), ("g1_43", 16)])
def test_self_collision_vs_oracle_and_reference(robot, n):
    rm = load_robot(robot)
    q = random_q(rm, n, seed=23)
    _, sph, _, _ = O.fk_forward(rm, q)
    want_c, want_g, want_k = O.self_collision(sph, rm.sphere_padding, rm.collision_pairs, 5000.0)
    assert (want_c > 0).sum() > 0
    cost = SelfCollisionCost(rm, 5000.0, DEV)
    st = T(sph.reshape(n, 1, -1, 4)).requires_grad_(True)
    d = cost.forward(st)
    got_c = d.detach().cpu().numpy().reshape(n)
    np.testing.assert_allclose(got_c, want_c, rtol=1e-4, atol=1e-6 * want_c.max())
    got_g = cost._out_vec.cpu().numpy().reshape(want_g.shape)
    # identical worst pair (no exact ties on random inputs) -> identical sparsity pattern
    assert ((np.abs(got_g).sum(-1) > 0) == (np.abs(want_g).sum(-1) > 0)).all()
    grad_close(got_g, want_g)
    d.sum().backward()
    grad_close(st.grad.cpu().numpy().reshape(want_g.shape), want_g)
    if ref_kernels.comparing():
        def reference():
            d, v = ref_kernels.self_collision(rm, T(sph.reshape(n, 1, -1, 4)), cost.sphere_padding, cost.pairs, 5000.0)
            return d.view(n), v.view(want_g.shape)
        r = ref_kernels.recorded(("parity", "self_collision", robot, n), reference, whole=True)   # sparse: every row
        np.testing.assert_allclose(r.at(0, got_c), r[0], rtol=1e-4, atol=1e-6 * want_c.max())
        grad_close(r.at(1, got_g), r[1])
        np.testing.assert_allclose(r.at(0, want_c), r[0], rtol=1e-4, atol=1e-6 * want_c.max())


def test_self_collision_lazy_zeroing_and_golden():
    """Second call on different spheres must clear the two rows the first call wrote
    (sparse_index protocol, self_collision_helper.cuh:151-192)."""
    g = np.load(os.path.join(GOLD, "franka_fk_self_b64.npz"))
    rm = load_robot("franka")
    cost = SelfCollisionCost(rm, 5000.0, DEV)
    sph = g["spheres"].reshape(64, 1, -1, 4)
    d1 = cost.forward(T(sph).requires_grad_(True)).detach().cpu().numpy().reshape(-1)
    np.testing.assert_allclose(d1, g["self_cost"], rtol=1e-4, atol=1e-3)
    grad_close(cost._out_vec.cpu().numpy().reshape(g["self_grad"].shape), g["self_grad"])
    d2 = cost.forward(T(sph[::-1].copy()).requires_grad_(True))
    grad_close(cost._out_vec.cpu().numpy().reshape(g["self_grad"].shape), g["self_grad"][::-1])
    assert int(cost._sparse.sum()) == 2 * int((g["self_cost"] > 0).sum())
    # disabled spheres (negative padded radius) never collide
    sph_off = sph.copy()
    sph_off[..., 3] = -1.0
    assert float(cost.forward(T(sph_off).requires_grad_(True)).abs().sum()) == 0.0
    assert float(cost._out_vec.abs().sum()) == 0.0


# ------------------------------------------------------------------------------------------------
def _scene(cub=None, vox=None):
    return SceneData(CuboidData.from_world(cub, DEV) if cub is not None else None,
                     VoxelData.from_world(vox, DEV) if vox is not None else None)


def _run_scene(sph, scene, w, eta, sweep=False, speed_dt=None, env=None, multi=False):
    B, H, S, _ = sph.shape
    buf = CollisionBuffer.from_shape(sph.shape, DEV)
    wt, et = T(np.array([w], np.float32)), T(np.array([eta], np.float32))
    st = T(sph).requires_grad_(True)
    eq = T(env) if env is not None else torch.zeros(B, dtype=torch.int32, device=DEV)
    if sweep:
        dt = T(np.array([speed_dt if speed_dt else 0.0], np.float32))
        d = SweptSphereObstacleCollision.apply(st, buf, scene, wt, et, None, dt, speed_dt is not None, eq, multi, False)
    else:
        d = SphereObstacleCollision.apply(st, buf, scene, wt, et, None, eq, multi, False)
    d.sum().backward()
    return d.detach().cpu().numpy(), buf.gradient.cpu().numpy(), st.grad.cpu().numpy()


@pytest.mark.parametrize("case", cases(), ids=lambda c: c[0])
def test_voxel_property_cases_gpu(case):
    name, world, spheres, eta, sweep, check = case
    scene = _scene(vox=world)
    if sweep == "both":
        c0, g0, _ = _run_scene(spheres[:, :1], scene, 1.0, eta)
        c1, g1, _ = _run_scene(spheres, scene, 1.0, eta, sweep=True)
        np.testing.assert_allclose(c1, np.broadcast_to(c0, c1.shape), rtol=1e-6)
        np.testing.assert_allclose(g1, np.broadcast_to(g0, g1.shape), rtol=1e-6, atol=1e-7)
        return
    c, g, _ = _run_scene(spheres, scene, 1.0, eta, sweep=bool(sweep))
    assert check(c, g), (name, c, g)


def test_empty_scene_zero_and_cuboid_world():
    """tests/_src/cost/test_cost_scene_collision.py:265,298: empty scene -> 0; cuboids -> cost + gradient."""
    rm = load_robot("franka")
    q = random_walk_q(rm, 16, 4, seed=31)
    _, sph, _, _ = O.fk_forward(rm, q.reshape(-1, 7))
    sph = sph.reshape(16, 4, -1, 4)
    empty = CuboidWorld.create([], max_n=10)
    c, g, _ = _run_scene(sph, _scene(cub=empty), 100.0, 0.01)
    assert c.sum() == 0 and np.abs(g).sum() == 0
    cub = make_benchmark_cuboid_world()
    c, g, gi = _run_scene(sph, _scene(cub=cub), 100.0, 0.01)
    wc, wg = O.scene_collision(sph, 100.0, 0.01, cub, None)
    assert (wc > 0).sum() > 0
    np.testing.assert_allclose(c, wc, rtol=1e-4, atol=1e-6 * wc.max())
    grad_close(g, wg)
    grad_close(gi, wg)


@pytest.mark.parametrize("mode", ["discrete", "swept", "swept_speed"])
@pytest.mark.parametrize("world", ["cuboid", "voxel", "both"])
def test_scene_collision_vs_oracle(mode, world):
    rng = np.random.default_rng(0)
    B, H, S = 12, 10, 50
    pos = rng.uniform(-1.4, 1.4, size=(B, 1, S, 3)) + np.cumsum(rng.normal(0, 0.05, size=(B, H, S, 3)), axis=1)
    rad = rng.uniform(0.01, 0.12, size=(B, 1, S, 1))
    rad[:, :, ::9] = -1.0
    sph = np.concatenate([pos, np.broadcast_to(rad, (B, H, S, 1))], -1).astype(np.float32)
    cub = CuboidWorld.create([
        {"dims": [2.2, 2.2, 0.2], "pose": [0, 0, -0.1, 1, 0, 0, 0]},
        {"dims": [0.3, 0.4, 1.5], "pose": [0.45, 0.1, 0.3, 0.9238795, 0, 0.3826834, 0]}], max_n=10) if world != "voxel" else None
    vox = small_voxel_world() if world != "cuboid" else None
    sweep = mode != "discrete"
    dt = 0.05 if mode == "swept_speed" else None
    c, g, _ = _run_scene(sph, _scene(cub, vox), 5000.0, 0.02, sweep=sweep, speed_dt=dt)
    wc, wg = O.scene_collision(sph, 5000.0, 0.02, cub, vox, sweep=sweep, speed_dt=dt)
    assert (wc > 0).sum() > 50
    np.testing.assert_allclose(c, wc, rtol=1e-4, atol=1e-5 * wc.max())
    grad_close(g, wg, rtol=2e-3, scale=2e-5)


def test_swept_golden_fixture_and_multi_env():
    g = np.load(os.path.join(GOLD, "franka_swept_b4_h12.npz"))
    cub, vox = make_benchmark_cuboid_world(), small_voxel_world()
    c, gr, _ = _run_scene(g["spheres"], _scene(cub, vox), 100000.0, 0.0025, sweep=True, speed_dt=0.05)
    np.testing.assert_allclose(c, g["scene_cost"], rtol=1e-4, atol=1e-5 * g["scene_cost"].max())
    grad_close(gr, g["scene_grad"], rtol=2e-3, scale=2e-5)
    # two environments: env 1 has no obstacles
    cub2 = CuboidWorld.create([{"dims": [2.2, 2.2, 0.2], "pose": [0, 0, -0.1, 1, 0, 0, 0]}], max_n=4, num_envs=2)
    cub2.count[1] = 0
    env = np.array([0, 1, 0, 1], np.int32)
    c2, _, _ = _run_scene(g["spheres"], _scene(cub=cub2), 10.0, 0.01, env=env, multi=True)
    wc, _ = O.scene_collision(g["spheres"], 10.0, 0.01, cub2, None, env_query_idx=env)
    np.testing.assert_allclose(c2, wc, rtol=1e-4, atol=1e-6)
    assert c2[1].sum() == 0 and c2[3].sum() == 0


# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lie", [False, True])
def test_tool_pose_vs_oracle(lie):
    rng = np.random.default_rng(9)
    B, H, L, G, NG = 10, 5, 3, 4, 3
    pos = rng.normal(size=(B, H, L, 3)).astype(np.float32)
    quat = rng.normal(size=(B, H, L, 4)).astype(np.float32)
    quat /= np.linalg.norm(quat, axis=-1, keepdims=True)
    gpos = rng.normal(size=(G, L, NG, 3)).astype(np.float32)
    gquat = rng.normal(size=(G, L, NG, 4)).astype(np.float32)
    gquat /= np.linalg.norm(gquat, axis=-1, keepdims=True)
    idx = rng.integers(0, G, size=(B, 1)).astype(np.int32)
    w = np.array([1000.0, 30.0], np.float32)
    at = rng.uniform(0.2, 1.5, size=(L, 6)).astype(np.float32)
    ant = rng.uniform(0.0, 1.0, size=(L, 6)).astype(np.float32)
    tt = np.full((L, 2), 1e-3, np.float32)
    tnt = np.full((L, 2), 1e-2, np.float32)
    z = lambda *s, dt=torch.float32: torch.zeros(s, dtype=dt, device=DEV)  # noqa: E731
    od, opd, ord_, opg, org, ogi = z(B, H, 2 * L), z(B, H, L), z(B, H, L), z(B, H, L, 3), z(B, H, L, 4), z(B, H, L, dt=torch.int32)
    cb_cost.tool_pose_distance(T(pos), T(quat), T(gpos), T(gquat), T(idx), T(w), T(at), T(ant), T(tt), T(tnt),
                               torch.zeros(L, dtype=torch.uint8, device=DEV), od, opd, ord_, opg, org, ogi, use_lie_group=lie)
    c, gp, gq, gi, pe, re = O.tool_pose_cost(pos, quat, gpos, gquat, idx[:, 0], w, at, ant, tt, tnt, use_lie_group=lie)
    assert (ogi.cpu().numpy() == gi).all()
    np.testing.assert_allclose(od.cpu().numpy(), c, rtol=2e-4, atol=1e-4 * c.max())
    grad_close(opg.cpu().numpy(), gp)
    grad_close(org.cpu().numpy(), gq, rtol=2e-3, scale=1e-4)
    np.testing.assert_allclose(opd.cpu().numpy(), pe, rtol=2e-4, atol=1e-5)
    np.testing.assert_allclose(ord_.cpu().numpy(), re, rtol=2e-4, atol=1e-5)


def test_cspace_costs_vs_oracle():
    rm = load_robot("franka")
    rng = np.random.default_rng(3)
    B, H, D = 9, 7, 7
    q = rng.uniform(rm.position_limits[0] - 0.15, rm.position_limits[1] + 0.15, size=(B, H, D)).astype(np.float32)
    v, a, j = [rng.normal(0, s, size=(B, H, D)).astype(np.float32) for s in (2.0, 12.0, 400.0)]
    dt = rng.uniform(0.02, 0.2, size=B).astype(np.float32)
    lim = dict(p=rm.position_limits, v=rm.velocity_limits, a=rm.acceleration_limits, j=rm.jerk_limits, tau=rm.effort_limits)
    w = np.array([10000.0, 10000.0, 100.0, 50.0, 100.0], np.float32)
    act = np.full(5, 0.01, np.float32)
    reg = np.array([1000.0, 10000.0, 5.0, 0.0, 0.0], np.float32)
    tgt = random_q(rm, 2, seed=8)
    it = (np.arange(B) % 2).astype(np.int32)
    want_c, want_g = O.cspace_state_cost(q, v, a, j, dt, lim, w, act, reg, True, True, target=tgt, idxs_target=it,
                                         target_weight=3.0, non_terminal_factor=0.5, target_dof_weight=np.ones(D))
    z = lambda: torch.zeros((B, H, D), dtype=torch.float32, device=DEV)  # noqa: E731
    oc, gp, gv, ga, gj, gt = z(), z(), z(), z(), z(), z()
    cb_cost.cspace_state_cost(T(q), T(v), T(a), T(j), z(), T(dt), T(tgt), T(it), T(lim["p"]), T(lim["v"]), T(lim["a"]),
                              T(lim["j"]), T(lim["tau"]), T(w), T(act), T(reg), T(np.array([3.0], np.float32)),
                              T(np.array([0.5], np.float32)), T(np.ones(D, np.float32)), oc, gp, gv, ga, gj, gt, True, True)
    np.testing.assert_allclose(oc.cpu().numpy(), want_c, rtol=2e-4, atol=1e-5 * want_c.max())
    for got, want in zip((gp, gv, ga, gj), want_g[:4]):
        grad_close(got.cpu().numpy(), want)
    # POSITION (IK) variant
    wp = np.array([5000.0, 0.0], np.float32)
    ap = np.array([0.01, 0.01], np.float32)
    want_c, want_g = O.cspace_position_cost(q, rm.position_limits, wp, ap)
    oc, gp, gt = z(), z(), z()
    zi = torch.zeros(B, dtype=torch.int32, device=DEV)
    zd = torch.zeros((1, D), dtype=torch.float32, device=DEV)
    cb_cost.cspace_position_cost(T(q), z(), zd, zi, T(rm.position_limits), T(rm.effort_limits), T(wp), T(ap),
                                 T(np.array([0.0], np.float32)), T(np.ones(D, np.float32)), T(np.zeros(2, np.float32)),
                                 zd, zd, zi, T(rm.velocity_limits), torch.zeros(1, dtype=torch.float32, device=DEV), oc, gp, gt)
    assert want_c.max() > 0
    np.testing.assert_allclose(oc.cpu().numpy(), want_c, rtol=2e-4, atol=1e-6 * want_c.max())
    grad_close(gp.cpu().numpy(), want_g)
