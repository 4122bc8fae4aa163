"""The GPU test-suite, re-run without a GPU: the test FUNCTIONS of tests/test_gpu_*.py are called here with `DEV = "cpu"` against the
product library compiled for the host SIMT emulation (tests/simt: every translation unit of curobo_b200/csrc as C++, CTA threads
and warp lanes played by std::threads, the product's own cb200_* entry points and launch logic).  The Python host layer is the
product's, unmodified; the swap consists of (1) curobo_b200.lib.load returning the emulated library and (2)
backends.tensor_checks.require_cuda / _stream_of being neutralised -- both exist only inside this fixture.  Full-size property tests,
CUDA-graph captures and the comparisons with the reference's compiled CUDA kernels need a real GPU and are not re-run.

This is what value-checks, before any B200 time is spent on them, the GPU tests that were written after the last GPU session
(files test_gpu_zx_*, zy_*, zz_*)."""
import ctypes as C
import importlib
import os
import subprocess

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIMT = os.path.join(ROOT, "tests", "simt")
UNITS = ["simt_kernels.cpp", "simt_trajectory_abi.cpp", "simt_dynamics.cpp", "simt_edt.cpp", "simt_optim_abi.cpp"]


@pytest.fixture(scope="module")
def emulated_library():
    from curobo_b200 import lib as cblib
    tsan = os.environ.get("CB200_SIMT_TSAN") == "1"   # race-detector build: run pytest with LD_PRELOAD=libtsan.so (see below)
    so = os.path.join(SIMT, "libsimt_full_tsan.so" if tsan else "libsimt_full.so")
    csrc = os.path.join(ROOT, "curobo_b200", "csrc")
    deps = [os.path.join(SIMT, u) for u in UNITS] + [os.path.join(SIMT, h) for h in ("cuda_runtime.h", "cuda_fp16.h")] + \
        [os.path.join(csrc, f) for f in sorted(os.listdir(csrc))]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.run(["g++", "-std=c++20", "-O1", "-pthread", "-shared", "-fPIC", "-w", *(["-g", "-fsanitize=thread"] if tsan else []),
                        "-I", SIMT, *[os.path.join(SIMT, u) for u in UNITS], "-o", so], check=True)
    L = C.CDLL(so)
    for name, (args, res) in cblib._SIGS.items():
        fn = getattr(L, name)                     # every ABI symbol must exist in the emulated library too
        fn.argtypes, fn.restype = args, res
    assert L.cb200_abi_version() == 6
    return L


@pytest.fixture
def run(monkeypatch, emulated_library):
    from curobo_b200 import lib as cblib
    from curobo_b200.backends import tensor_checks as tc
    import ref_kernels
    monkeypatch.setattr(cblib, "_LIB", emulated_library)
    monkeypatch.setattr(cblib, "load", lambda: emulated_library)
    monkeypatch.setattr(tc, "require_cuda", lambda device, message: None)
    monkeypatch.setattr(tc, "_stream_of", lambda device: 0)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    monkeypatch.setattr(torch.cuda, "is_current_stream_capturing", lambda: False)
    monkeypatch.setattr(ref_kernels, "available", lambda: False)
    monkeypatch.setattr(ref_kernels, "comparing", lambda: False)

    def call(module, test, *args, **kwargs):
        mod = importlib.import_module(module)
        monkeypatch.setattr(mod, "DEV", "cpu")
        if hasattr(mod, "T") and not getattr(mod.T, "_copies", False):
            orig = mod.T                          # torch.as_tensor(x).to("cpu") aliases the numpy input; on a GPU .to() copies

            def T(a, *r, **k):
                return orig(np.array(a, copy=True), *r, **k)
            T._copies = True
            monkeypatch.setattr(mod, "T", T)
        return getattr(mod, test)(*args, **kwargs)
    return call


# ------------------------------------------------------------------------------------------------ drop-in operators
@pytest.mark.parametrize("robot,n", [("franka", 64), ("g1_29", 12)])
def test_fk_forward(run, robot, n):
    run("test_gpu_parity", "test_fk_forward_vs_oracle_and_reference", robot, n)


def test_fk_misc(run):
    run("test_gpu_parity", "test_fk_without_spheres_entry_point")
    run("test_gpu_parity", "test_fk_golden_vector_on_gpu")
    run("test_gpu_parity", "test_fk_forward_golden_fixture")
    run("test_gpu_parity", "test_fk_multi_sphere_configs")


@pytest.mark.parametrize("robot,n,sparse", [("franka", 40, False), ("franka", 40, True), ("g1_29", 8, True)])
def test_fk_backward(run, robot, n, sparse):
    run("test_gpu_parity", "test_fk_backward_vs_oracle_and_reference", robot, n, sparse)
    if robot == "franka" and not sparse:
        run("test_gpu_parity", "test_fk_backward_mimic_and_negative_axis")


@pytest.mark.parametrize("robot,n", [("franka", 48), ("g1_29", 6)])
def test_self_collision(run, robot, n):
    run("test_gpu_parity", "test_self_collision_vs_oracle_and_reference", robot, n)


def test_self_collision_lazy_zeroing(run):
    run("test_gpu_parity", "test_self_collision_lazy_zeroing_and_golden")


@pytest.mark.parametrize("mode", ["discrete", "swept", "swept_speed"])
@pytest.mark.parametrize("world", ["cuboid", "voxel", "both"])
def test_scene_collision(run, mode, world):
    run("test_gpu_parity", "test_scene_collision_vs_oracle", mode, world)


def test_scene_misc(run):
    run("test_gpu_parity", "test_empty_scene_zero_and_cuboid_world")
    run("test_gpu_parity", "test_swept_golden_fixture_and_multi_env")
    mod = importlib.import_module("test_gpu_parity")
    for case in mod.cases():
        run("test_gpu_parity", "test_voxel_property_cases_gpu", case)


@pytest.mark.parametrize("lie", [False, True])
def test_tool_pose(run, lie):
    run("test_gpu_parity", "test_tool_pose_vs_oracle", lie)


def test_cspace_costs(run):
    run("test_gpu_parity", "test_cspace_costs_vs_oracle")


# ------------------------------------------------------------------------------------------------ fused rollout
def test_fused_ik(run):
    run("test_gpu_rollout", "test_franka_ik_rollout_vs_oracle_and_golden")
    if os.environ.get("CB200_EMULATE_LONG") == "1":
        run("test_gpu_rollout", "test_franka_ik_rollout_larger_batch")
    run("test_gpu_rollout", "test_franka_esdf_horizon_rollout_terminal_weights")
    run("test_gpu_rollout", "test_state_cspace_rollout_vs_oracle")


@pytest.mark.parametrize("B,H,speed", [(4, 12, True), (5, 5, False), (6, 1, True), (3, 9, True)])
def test_fused_trajectory(run, B, H, speed):
    run("test_gpu_rollout", "test_traj_rollout_vs_oracle", B, H, speed)


@pytest.mark.parametrize("B,H,with_dofw", [(5, 30, True), (3, 7, False), (4, 1, True)])
def test_fused_mpc_config(run, B, H, with_dofw):
    run("test_gpu_rollout", "test_mpc_config_rollout_vs_oracle", B, H, with_dofw)


def test_fused_position_target_and_sphere_configs(run):
    run("test_gpu_rollout", "test_ik_position_cspace_target_vs_oracle")
    run("test_gpu_rollout", "test_fused_rollout_sphere_configs", "discrete")
    run("test_gpu_rollout", "test_fused_rollout_sphere_configs", "swept")


def test_rollout_protocol_adapter(run):
    run("test_gpu_rollout_protocol", "test_protocol_surface")
    run("test_gpu_rollout_protocol", "test_ik_rollout_through_optimizer_contract_vs_oracle")
    run("test_gpu_rollout_protocol", "test_mpc_position_actions_with_state")
    run("test_gpu_rollout_protocol", "test_bspline_action_space_gradient_wrt_knots")


@pytest.mark.parametrize("robot,n", [("g1_29", 6), ("g1_43", 4)])
def test_fused_humanoid(run, robot, n):
    run("test_gpu_rollout", "test_humanoid_esdf_rollout_vs_oracle", robot, n)


@pytest.mark.parametrize("mode", ["discrete", "swept"])
def test_fused_multi_env(run, mode):
    run("test_gpu_rollout", "test_fused_rollout_multi_env", mode)


@pytest.mark.parametrize("lie", [False, True])
def test_fused_goalset_and_tool_frames(run, lie):
    run("test_gpu_rollout", "test_fused_rollout_goalset_and_tool_frames", lie)


def test_fused_voxel_mip(run):
    run("test_gpu_rollout", "test_voxel_mip_build_and_exact_cull")


# ------------------------------------------------------------------------------------------------ B-spline, optimizer, dynamics
def test_bspline(run):
    mod = importlib.import_module("test_gpu_bspline")
    for kw in mod.CASES[::2]:                      # every other case: all three degrees, both boundary modes
        run("test_gpu_bspline", "test_forward_vs_oracle_and_reference", kw)
        run("test_gpu_bspline", "test_backward_vs_oracle_and_reference", kw)
    run("test_gpu_bspline", "test_single_dt_vs_oracle_and_reference")
    # test_error_behaviour checks that host tensors are refused: exactly the rule this fixture switches off
    for implicit in (False, True):
        run("test_gpu_bspline", "test_autograd_function_and_state_transition", implicit)


@pytest.mark.parametrize("mode", ["trajopt_swept", "discrete"])
@pytest.mark.parametrize("degree,steps,implicit", [(4, 4, False), (3, 2, True), (5, 1, False)])
def test_fused_knots(run, mode, degree, steps, implicit):
    run("test_gpu_bspline", "test_fused_knots_rollout_vs_oracle_chain", mode, degree, steps, implicit)


def test_optimizer_kernels(run):
    mod = importlib.import_module("test_gpu_optim")
    long = os.environ.get("CB200_EMULATE_LONG") == "1"
    for kw in (mod.LBFGS_CASES if long else mod.LBFGS_CASES[::3]):
        run("test_gpu_optim", "test_lbfgs_step_vs_oracle_and_reference", kw)
    for i, kw in enumerate(mod.LS_CASES if long else mod.LS_CASES[::2]):
        for strong, approx in (((False, True), (False, False), (True, False)) if long else [((False, True), (False, False), (True, False))[i % 3]]):
            run("test_gpu_optim", "test_line_search_vs_oracle_and_reference", kw, strong, approx)
    run("test_gpu_optim", "test_lbfgs_autograd_function_and_search_points")
    run("test_gpu_optim", "test_lbfgs_opt_solves_quadratics")


@pytest.mark.parametrize("robot,B,seed", [("franka", 9, 1), ("g1_29", 5, 2), ("g1_43", 3, 3), ("franka", 200, 4)])
def test_rnea(run, robot, B, seed):
    run("test_gpu_dynamics", "test_rnea_vs_oracle_and_reference", robot, B, seed)


@pytest.mark.parametrize("robot,B", [("franka", 2), ("g1_29", 37)])
def test_rnea_external_wrenches(run, robot, B):
    run("test_gpu_dynamics", "test_rnea_external_wrenches", robot, B)


def test_rnea_row_kernels(run, monkeypatch):
    run("test_gpu_dynamics", "test_rnea_row_kernels_match_cta_kernels", monkeypatch)


# ------------------------------------------------------------------------------------------------ written after the last GPU session
def test_pending_rnea_trees(run, monkeypatch):
    mod = importlib.import_module("test_gpu_zx_dynamics_trees")
    from dynamics_cases import RANDOM_TREES
    for nl, B, seed, mimic in RANDOM_TREES + [(23, 70, 41, True)]:
        for rows in (False, True):
            with monkeypatch.context() as m:
                run("test_gpu_zx_dynamics_trees", "test_rnea_on_random_trees", nl, B, seed, mimic, rows, m)
    for robot, B in (("franka", 100), ("g1_29", 70)):
        for R in (8, 16, 32):
            with monkeypatch.context() as m:
                run("test_gpu_zx_dynamics_trees", "test_rnea_every_rows_per_cta_variant", robot, B, R, m)
    assert mod.DEV == "cpu"


@pytest.mark.parametrize("robot,B,H", [("franka", 6, 5), ("g1_29", 3, 4)])
def test_pending_dynamics_state_cost(run, robot, B, H):
    run("test_gpu_zy_effort_cost", "test_dynamics_state_cost_vs_oracle", robot, B, H)


@pytest.mark.parametrize("robot,n,buried", [("g1_29", 5, False), ("g1_29", 3, True), ("franka", 6, True)])
def test_big_robot_kernel(run, monkeypatch, robot, n, buried):
    run("test_gpu_rollout", "test_big_robot_kernel_matches_standard_kernel_and_oracle", monkeypatch, robot, n, buried)


def test_traj_dense_gradients_over_many_tiles(run, monkeypatch):
    run("test_gpu_rollout", "test_traj_dense_gradients_over_many_tiles", monkeypatch, 40, 20)


@pytest.mark.parametrize("robot,n,team,scene", [("g1_29", 5, 2, "esdf"), ("g1_29", 3, 4, "both"), ("g1_29", 3, 2, "buried"),
                                                 ("franka", 6, 4, "cuboid")])
def test_team_kernel(run, monkeypatch, robot, n, team, scene):
    run("test_gpu_rollout", "test_team_kernel_matches_big_kernel_and_oracle", monkeypatch, robot, n, team, scene)


@pytest.mark.skipif(not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "pyref", "MANIFEST.json")),
                    reason="oracle/_ref/pyref not built")
def test_reference_call_sites_over_b200_backend(run):
    """The reference's own autograd Functions (byte code under oracle/_ref/pyref) over curobo_b200.backends, here over the emulated
    library: the same test functions the GPU box runs (tests/test_gpu_reference_callsites.py)."""
    mod = importlib.import_module("test_gpu_reference_callsites")
    ref = mod.load_reference()
    run("test_gpu_reference_callsites", "test_reference_kinematics_function_over_b200_backend", ref, "franka", 16)
    run("test_gpu_reference_callsites", "test_reference_self_collision_function_over_b200_backend", ref, "franka", 12)
    run("test_gpu_reference_callsites", "test_reference_bspline_function_over_b200_backend", ref, True)
    run("test_gpu_reference_callsites", "test_reference_lbfgs_function_over_b200_backend", ref)
    # the reference's optimizer on top of the Rollout-protocol adapter (25 iterations, 6 problems here; 100 x 24 on the GPU)
    run("test_gpu_reference_callsites", "test_reference_lbfgs_optimizer_drives_the_b200_rollout", ref, 25, 6)


def test_mesh_obstacles(run):
    """Mesh obstacles through the emulated mesh_collision_kernel: box mesh == cuboid (the reference's regression), brute-force
    oracle, mesh + cuboid accumulation / multi-env / disabled slots."""
    run("test_gpu_mesh", "test_box_mesh_costs_what_the_cuboid_costs", False)
    run("test_gpu_mesh", "test_box_mesh_costs_what_the_cuboid_costs", True)
    run("test_gpu_mesh", "test_mesh_collision_vs_brute_force_oracle", "icosphere")
    run("test_gpu_mesh", "test_mesh_collision_vs_brute_force_oracle", "box")
    run("test_gpu_mesh", "test_mesh_with_cuboids_multi_env_and_disabled_slots")


def test_pending_edt(run):
    mod = importlib.import_module("test_gpu_zz_edt")
    from edt_cases import MEDIUM, SMALL
    for kind, shape, p in SMALL + MEDIUM[:4]:
        run("test_gpu_zz_edt", "test_nearest_site_transform_is_exact", kind, shape, p)
    run("test_gpu_zz_edt", "test_operator_argument_checks_emulated") if hasattr(mod, "test_operator_argument_checks_emulated") else None
    for shape, skip in (((24, 20, 28), 1.0), ((16, 16, 16), 0.0), ((20, 31, 12), 2.0)):
        run("test_gpu_zz_edt", "test_dense_esdf_builder_vs_oracle", shape, skip)


def test_gather_seeding_kernel_vs_reference_source_golden(run, monkeypatch):
    """cb200_esdf_seed_sites_gather (the reference's DEFAULT seeding, seed_esdf_sites_gather_kernel) against the output of the
    reference's kernel source under the Warp stand-in, and DenseESDFBuilder(seeding_method="gather") end to end against the oracle.
    Emulated only: the kernel was written after the round's GPU budget was spent (its arithmetic is spelled with IEEE intrinsics,
    so the B200 must give the same voxels); the builder's default stays "scatter", which is GPU-validated."""
    from oracle import edt_oracle as E
    from curobo_b200.backends import pba as pba_cu
    from curobo_b200.esdf import DenseESDFBuilder
    g = np.load(os.path.join(ROOT, "tests", "golden", "esdf_reference_golden.npz"))
    shape = tuple(int(v) for v in g["shape"])
    voxel, trunc, minw = float(g["voxel"]), float(g["trunc"]), float(g["min_weight"])
    static = g["static"].astype(np.float32)
    static_in = np.where(np.isfinite(static), static, np.float32(1e10)).astype(np.float32)
    comb = E.tsdf_combined_sdf(g["block_data"], static_in, minw)
    sites = torch.empty(int(np.prod(shape)), dtype=torch.int32)
    pba_cu.launch_esdf_seed_sites_gather(torch.as_tensor(comb).view(-1), sites, *shape, voxel, trunc, g["origin"])
    assert np.array_equal(sites.numpy().reshape(shape), g["seeds_gather"])
    b = DenseESDFBuilder(shape, voxel, trunc, "cpu", seeding_method="gather", origin=g["origin"])
    field = b.compute(torch.as_tensor(comb), torch.as_tensor(static_in)).numpy().astype(np.float32)
    res = b.site_index.numpy()
    seeds = E.seed_sites_gather_from_sdf(comb, voxel, trunc, g["origin"])
    assert np.array_equal(E.squared_distance(res), E.squared_distance(E.pba3d(seeds, "zyx")))
    want = E.signed_distance_fp16(res, static_in, comb, voxel, 1.0).astype(np.float32)
    assert np.array_equal(np.sign(field), np.sign(want)) and np.abs(field - want).max() <= 2e-3
    with pytest.raises(ValueError):
        DenseESDFBuilder(shape, voxel, trunc, "cpu", seeding_method="nearest")


def test_stamp_cuboids_kernel_vs_reference_source_golden(run, monkeypatch):
    """cb200_tsdf_stamp_cuboids (dense form of the reference's stamp_sdf_kernel) against the output of the reference's kernel source
    under the Warp stand-in, through DenseTSDF.stamp_cuboids; then world cuboids + depth images -> ESDF end to end against the
    oracle.  Emulated only (written after the round's GPU budget was spent); nothing on the GPU path depends on it."""
    from oracle import edt_oracle as E
    from curobo_b200.esdf import DenseESDFBuilder, DenseTSDF
    from curobo_b200.scene import CuboidData
    from curobo_b200.world import CuboidWorld
    g = np.load(os.path.join(ROOT, "tests", "golden", "esdf_reference_golden.npz"))
    t = np.load(os.path.join(ROOT, "tests", "golden", "tsdf_reference_golden.npz"))
    shape = tuple(int(v) for v in g["shape"])
    voxel, trunc, minw = float(g["voxel"]), float(g["trunc"]), float(g["min_weight"])
    cw = CuboidWorld(g["cub_dims"], g["cub_inv_pose"], g["cub_enable"], g["cub_count"])
    cd = CuboidData.from_world(cw, "cpu")
    tsdf = DenseTSDF(shape, voxel, trunc, "cpu", origin=g["origin"], depth_min=float(t["a/depth_min"]),
                     depth_max=float(t["a/depth_max"]), minimum_tsdf_weight=minw)
    for env in (0, 1):
        st = tsdf.stamp_cuboids(cd, env).numpy()
        want = g["stamped"][env].astype(np.float32)
        m = np.isfinite(want)
        assert np.array_equal(st < 1e9, m) and np.abs(st[m] - want[m]).max() <= 2e-4
    for _ in range(2):
        tsdf.integrate(torch.as_tensor(t["a/depth"]), torch.as_tensor(t["a/K"]), torch.as_tensor(t["a/pos"]), torch.as_tensor(t["a/quat"]))
    assert np.array_equal(tsdf.block_data.numpy(), t["a/block_data"][-1])
    comb = tsdf.combined_sdf(tsdf.static_sdf).numpy()
    assert np.array_equal(comb, E.tsdf_combined_sdf(t["a/block_data"][-1], st, minw))
    b = DenseESDFBuilder(shape, voxel, trunc, "cpu", seeding_method="gather", origin=g["origin"])
    field = b.compute(torch.as_tensor(comb), tsdf.static_sdf).numpy().astype(np.float32)
    want = E.signed_distance_fp16(b.site_index.numpy(), st, comb, voxel, 1.0).astype(np.float32)
    assert np.array_equal(np.sign(field), np.sign(want)) and np.abs(field - want).max() <= 2e-3 and (want < 0).sum() > 0
    tsdf.reset()
    assert float(tsdf.block_data.abs().sum()) == 0.0 and bool((tsdf.static_sdf > 1e9).all())


def test_built_esdf_feeds_the_collision_operator(run, monkeypatch):
    """World cuboid -> static TSDF channel -> ESDF (DenseESDFBuilder) -> VoxelData (to_voxel_data) -> SphereObstacleCollision: the
    cost of spheres against the BUILT grid agrees with their cost against the analytic cuboid to within a voxel, i.e. the producer's
    output is consumable by the hot path as it stands.  Emulated only (see test_stamp_cuboids_kernel_vs_reference_source_golden)."""
    import importlib
    from curobo_b200.esdf import DenseESDFBuilder, DenseTSDF
    from curobo_b200.scene import CollisionBuffer, CuboidData, SceneData, SphereObstacleCollision
    from curobo_b200.world import CuboidWorld
    shape, voxel = (40, 40, 40), 0.02
    trunc = 4 * voxel
    cw = CuboidWorld.create([{"dims": [0.3, 0.24, 0.2], "pose": [0.02, -0.01, 0.03, 1, 0, 0, 0]}])
    cd = CuboidData.from_world(cw, "cpu")
    tsdf = DenseTSDF(shape, voxel, trunc, "cpu")
    static = tsdf.stamp_cuboids(cd, 0)
    b = DenseESDFBuilder(shape, voxel, trunc, "cpu", seeding_method="gather")
    b.compute(static, static)
    vd = b.to_voxel_data(max_esdf_distance=10.0)
    assert vd.features.data_ptr() == b.dist_field.data_ptr()
    rng = np.random.default_rng(0)
    n = 400
    sph = np.zeros((1, 1, n, 4), np.float32)
    sph[0, 0, :, :3] = rng.uniform(-0.3, 0.3, size=(n, 3))
    sph[0, 0, :, 3] = 0.03
    w, eta = torch.tensor([1.0]), torch.tensor([0.05])
    costs = []
    for scene in (SceneData(cd, None), SceneData(None, vd)):
        buf = CollisionBuffer.from_shape((1, 1, n, 4), "cpu")
        costs.append(SphereObstacleCollision.apply(torch.as_tensor(sph), buf, scene, w, eta, None, torch.zeros(1, dtype=torch.int32),
                                                   False).numpy().reshape(-1).copy())
    exact, built = costs
    assert (exact > 0).sum() > 50 and (exact == 0).sum() > 50
    # (deep inside the box the static channel is unobserved -- |sdf| > truncation is not stamped -- and the ESDF measures from the
    #  truncation-boundary seeds, as in the reference; compare where the analytic distance is within the stamped band or outside)
    q = np.abs(sph[0, 0, :, :3] - np.array([0.02, -0.01, 0.03], np.float32)) - np.array([0.15, 0.12, 0.1], np.float32)
    sdf = np.linalg.norm(np.maximum(q, 0), axis=1) + np.minimum(q.max(1), 0)
    m = sdf > -(trunc - 2 * voxel)
    assert m.sum() > 300 and (exact[m] > 0).sum() > 30
    # the activation is 1-Lipschitz in the distance; the built field measures to the centres of a (dilated) band of seed voxels,
    # so it is within ~2 voxels of the analytic distance -- the reference's own approximation, not an error of the plumbing
    assert np.abs(exact[m] - built[m]).max() <= 2.5 * voxel, float(np.abs(exact[m] - built[m]).max())
    assert np.abs(exact[m] - built[m]).mean() <= 0.3 * voxel
    assert (built[~m] > 0).all(), "deep inside the box the built grid still reports a collision"


def test_depth_to_esdf_chain(run):
    run("test_gpu_zz_edt", "test_depth_to_esdf_chain_vs_oracle", (24, 24, 24))
    run("test_gpu_zz_edt", "test_depth_to_esdf_chain_vs_oracle", (40, 36, 44))
    run("test_gpu_zz_edt", "test_esdf_producer_kernels_vs_reference_source_goldens")


@pytest.mark.skipif(os.environ.get("CB200_EMULATE_LONG") != "1", reason="~5 min of emulated launches: set CB200_EMULATE_LONG=1 (passes)")
def test_complete_ik_solve(run):
    """24 goals x 16 seeds x 100 L-BFGS iterations, 3 kernel launches per iteration (step + search points, fused rollout on the
    expanded batch, line search + bookkeeping): >= 90 % of the goals solved to 5 mm -- every launch an emulated one."""
    run("test_gpu_optim", "test_ik_solve_end_to_end")


def test_bench_side_entries_execute(run, monkeypatch):
    """bench.py's `rnea` and `edt` entries (the `rnea` one died on a missing import in the last GPU session) executed end to end on
    tiny sizes against the emulated kernels, with CUDA events replaced by a dummy clock: no NameError / shape error left in them."""
    import sys
    sys.path.insert(0, ROOT)
    import bench

    class Event:
        def __init__(self, enable_timing=False): pass
        def record(self, *a): pass
        def elapsed_time(self, other): return 1.0

    monkeypatch.setattr(torch.cuda, "Event", Event)
    r = bench.rnea_bench("cpu", 6500.0, cases=(("franka", 64),), iters=2)
    assert set(r["franka_64"]) == {"forward", "backward"} and r["franka_64"]["forward"]["bytes_per_row"] == 4 * (4 * 7 + 13 * 20)
    e = bench.edt_bench("cpu", 6500.0, n=24, iters=1)
    assert e["grid"] == [24, 24, 24] and e["launches"] == 3 and e["sites"] > 0
    assert "error" not in e["depth_to_esdf"] and e["depth_to_esdf"]["observed_frac"] > 0.02, e["depth_to_esdf"]


@pytest.mark.parametrize("robot,B,H", [("franka", 3, 7), ("g1_29", 2, 4)])
def test_pending_dynamics_aware_rollout(run, robot, B, H):
    run("test_gpu_zy_effort_cost", "test_dynamics_aware_rollout_vs_oracle", robot, B, H)


def test_bench_dynamics_workloads_execute_and_agree(run):
    """bench.py's `<mpc>_dynamics` (torque inside the trajectory kernel) and `<mpc>_dynamics_host` (three extra launches) workloads,
    shrunk to two trajectories and a 64^3 ESDF: both build, run, and give the same costs and gradients."""
    import sys
    sys.path.insert(0, ROOT)
    import bench
    outs = {}
    for name in ("franka_mpc_1024x30_esdf_swept_dynamics", "franka_mpc_1024x30_esdf_swept_dynamics_host", "franka_mpc_1024x30_esdf_swept"):
        wl = bench.shard_workload(bench.make_workload(name), 0, 2)
        wl["voxel"]["n"], wl["voxel"]["voxel"] = 64, 0.04
        eng = bench.build_engine(wl, "cpu")
        kw = {k: torch.as_tensor(v) for k, v in wl["extra"].items()}
        o = eng.evaluate_action(torch.as_tensor(wl["q"]), **kw)
        outs[name] = (o.cost.clone(), o.grad_q.clone(), o.grad_vel.clone(), o.grad_acc.clone())
    f, h, plain = (outs[k] for k in outs)
    for a_, b_ in zip(f, h):
        assert torch.allclose(a_, b_, rtol=2e-3, atol=2e-5 * float(b_.abs().max()))
    # the effort terms are live in the dynamics workloads (which keep the trajopt weights; the plain MPC workload runs lbfgs_mpc.yml)
    assert float(f[0].sum()) > 0 and not torch.allclose(f[0], plain[0])


def test_pending_dynamics_aware_knots(run):
    run("test_gpu_zy_effort_cost", "test_dynamics_aware_knots_rollout_is_consistent")


@pytest.mark.parametrize("robot,n", [("franka", 33), ("g1_29", 9)])
def test_pending_center_of_mass(run, robot, n):
    run("test_gpu_zzz_center_of_mass", "test_center_of_mass_and_its_gradient", robot, n)
