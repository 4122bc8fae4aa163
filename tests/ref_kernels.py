"""The REFERENCE's own CUDA kernels as the GPU tests compare with them (test infrastructure only).

The tests read the kernels' outputs on each test's own inputs from tests/golden/reference_kernels_<group>.npz, recorded on a
B200 so that the comparison needs nothing outside this repository.  The launchers below are ctypes access to
oracle/_ref/libcurobo_ref.so, the reference's kernels compiled by `curobo_b200.build` from a checkout of the reference
(oracle/ref_kernels_launcher.cu); they are what records the fixtures, from the repository root on a GPU:

    CB200_RECORD_REFERENCE=<dir> python -m pytest -m gpu tests/test_gpu_parity.py tests/test_gpu_bspline.py \\
        tests/test_gpu_optim.py tests/test_gpu_dynamics.py tests/test_gpu_zz_edt.py tests/test_gpu_zzz_center_of_mass.py
    cp <dir>/reference_kernels_*.npz tests/golden/
"""
import ctypes as C
import json
import os

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PATH = os.path.join(ROOT, "oracle", "_ref", "libcurobo_ref.so")
GOLDEN = os.path.join(ROOT, "tests", "golden")
RECORD = os.environ.get("CB200_RECORD_REFERENCE")
BUDGET = 1024        # elements kept per leading-axis length in a recorded case (whole entries of that axis)


def available() -> bool:
    """Whether the reference's kernels themselves are at hand (oracle/_ref, built where the reference's sources are)."""
    return os.path.exists(PATH)


def comparing() -> bool:
    """Whether tests compare with the reference's kernels: always, through the recorded outputs.  The emulated GPU suite
    (tests/test_emulated_gpu_suite_cpu.py) turns it off: its host build of our kernels rounds differently from the device."""
    return True


def sample_rows(n, row_elems):
    """Entries kept of a leading axis of length n whose entries hold row_elems elements (summed over the outputs sharing
    the axis): all when they fit BUDGET, else the first, the last and a fixed seeded sample of the others."""
    k = max(2, BUDGET // max(1, row_elems))
    if n * row_elems <= BUDGET or k >= n:
        return np.arange(n)
    mid = np.random.default_rng(n).choice(np.arange(1, n - 1), k - 2, replace=False)
    return np.sort(np.concatenate([[0, n - 1], mid])).astype(np.int64)


class Recorded:
    """r[i]: the reference's output i at its kept entries of the leading axis; r.at(i, a): the same entries of an array
    `a` shaped like output i (ours, the oracle's); r.rows(i): their indices."""

    def __init__(self, outs, rows, shapes):
        self._outs, self._rows, self._shapes = outs, rows, shapes

    def __len__(self):
        return len(self._outs)

    def __getitem__(self, i):
        return self._outs[i]

    def rows(self, i):
        return self._rows[i]

    def at(self, i, a):
        assert tuple(np.shape(a)) == self._shapes[i], (np.shape(a), self._shapes[i])
        return np.asarray(a)[self._rows[i]]


def _read(path):
    """{case name: [(full shape, kept rows, values) per output]} of one fixture file: one concatenated array per dtype
    plus a JSON index (few archive members keep the file small)."""
    with np.load(path) as g:
        data = {k: g[k] for k in g.files}
    recs = {}
    for e in json.loads(str(data["index"])):
        shape, rows = tuple(e["shape"]), np.asarray(e["rows"], np.int64)
        v = data[e["dtype"]][e["offset"]:e["offset"] + e["count"]].reshape((len(rows),) + shape[1:])
        recs.setdefault(e["name"], []).append((shape, rows, v))
    return recs


def _write(path, recs):
    index, chunks, sizes = [], {}, {}
    for name, outs in recs.items():
        for shape, rows, v in outs:
            dt = v.dtype.name
            index.append({"name": name, "shape": list(shape), "rows": [int(r) for r in rows], "dtype": dt,
                          "offset": sizes.get(dt, 0), "count": v.size})
            chunks.setdefault(dt, []).append(v.reshape(-1))
            sizes[dt] = sizes.get(dt, 0) + v.size
    np.savez_compressed(path, index=np.array(json.dumps(index)), **{dt: np.concatenate(c) for dt, c in chunks.items()})


_golden = {}


def recorded(key, run, whole=False) -> Recorded:
    """The reference's outputs for one test case: key = (group, name parts...); run() launches the reference's kernels on
    the test's inputs and returns its outputs (a tensor or a sequence of them).  Outputs sharing a leading-axis length
    keep the same entries of it (sample_rows); whole=True keeps every entry (sparse outputs, where a sample would hold
    only zeros).  Replayed from tests/golden unless CB200_RECORD_REFERENCE names a directory: then run() is called and
    its kept outputs are added to <dir>/reference_kernels_<group>.npz."""
    group, name = key[0], "-".join(str(k) for k in key[1:])
    fname = f"reference_kernels_{group}.npz"
    if RECORD is None:
        if group not in _golden:
            _golden[group] = _read(os.path.join(GOLDEN, fname))
        if name not in _golden[group]:
            raise KeyError(f"no recorded reference output {name!r} in tests/golden/{fname}")
        outs = _golden[group][name]
        return Recorded([v for _, _, v in outs], [r for _, r, _ in outs], [s for s, _, _ in outs])
    outs = run()
    outs = [outs] if torch.is_tensor(outs) or isinstance(outs, np.ndarray) else list(outs)
    torch.cuda.synchronize()
    outs = [o.detach().cpu().numpy() if torch.is_tensor(o) else np.asarray(o) for o in outs]
    per_len = {}
    for o in outs:
        per_len[o.shape[0]] = per_len.get(o.shape[0], 0) + int(np.prod(o.shape[1:]))
    kept = {n: np.arange(n) if whole else sample_rows(n, e) for n, e in per_len.items()}
    rows = [kept[o.shape[0]] for o in outs]
    r = Recorded([o[k] for o, k in zip(outs, rows)], rows, [o.shape for o in outs])
    os.makedirs(RECORD, exist_ok=True)
    path = os.path.join(RECORD, fname)
    recs = _read(path) if os.path.exists(path) else {}
    recs[name] = [(o.shape, rows[i], r[i]) for i, o in enumerate(outs)]
    _write(path, recs)
    return r


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(PATH)
    return _lib


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _stream(dev):
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def fk_forward(kp, q, horizon=1, env_query_idx=None):
    """q [N,D] -> (link_pos, link_quat, spheres, cumul) through kinematics_forward_spheres_kernel."""
    dev = q.device
    N = q.shape[0]
    z = lambda *s: torch.zeros(s, dtype=torch.float32, device=dev)  # noqa: E731
    pos, quat = z(N, kp.num_pose_links, 3), z(N, kp.num_pose_links, 4)
    sph, com, cum = z(N, kp.num_spheres, 4), z(N, 4), z(N, kp.num_links, 3, 4)
    eq = env_query_idx if env_query_idx is not None else torch.zeros(1, dtype=torch.int32, device=dev)
    err = lib().ref_kinematics_forward_spheres(
        _p(pos), _p(quat), _p(sph), _p(com), _p(cum), _p(q), _p(kp.fixed_transforms), _p(kp.link_spheres),
        _p(kp.link_masses_com), _p(kp.joint_map_type), _p(kp.joint_map), _p(kp.link_map), _p(kp.tool_frame_map),
        _p(kp.link_sphere_idx_map), _p(kp.joint_offset_map), _p(eq), kp.num_envs, N, horizon, kp.num_dof,
        kp.num_spheres, kp.num_links, kp.num_pose_links, _stream(dev))
    assert err == 0, err
    return pos, quat, sph, cum


def fk_backward(kp, cumul, g_pos, g_quat, g_sph, horizon=1, env_query_idx=None):
    dev = cumul.device
    N = cumul.shape[0]
    out = torch.zeros((N, kp.num_dof), dtype=torch.float32, device=dev)
    com = torch.zeros((N, 4), dtype=torch.float32, device=dev)
    eq = env_query_idx if env_query_idx is not None else torch.zeros(1, dtype=torch.int32, device=dev)
    err = lib().ref_kinematics_backward(
        _p(out), _p(g_pos), _p(g_quat), _p(g_sph), _p(com), _p(com), None, _p(cumul), _p(kp.link_spheres),
        _p(kp.link_masses_com), _p(kp.link_map), _p(kp.joint_map), _p(kp.joint_map_type), _p(kp.tool_frame_map),
        _p(kp.link_sphere_idx_map), _p(kp.link_chain_data), _p(kp.link_chain_offsets), _p(kp.joint_links_data),
        _p(kp.joint_links_offsets), _p(kp.joint_affects_endeffector), _p(kp.joint_offset_map), _p(eq), kp.num_envs, N,
        horizon, kp.num_dof, kp.num_spheres, kp.num_links, kp.num_pose_links, _stream(dev))
    assert err == 0, err
    return out


def self_collision(rm, spheres, padding, pairs, weight):
    """spheres [B,H,S,4] -> (distance [B,H], grad [B,H,S,4]) through the reference kernels
    (single-kernel or map-reduce path chosen like the reference does)."""
    dev = spheres.device
    B, H, S, _ = spheres.shape
    nb = rm.num_blocks_per_batch
    dist = torch.zeros((B, H), dtype=torch.float32, device=dev)
    vec = torch.zeros((B, H, S, 4), dtype=torch.float32, device=dev)
    sparse = torch.zeros((B, H, S), dtype=torch.uint8, device=dev)
    pd = torch.zeros((1,), dtype=torch.float32, device=dev)
    bv = torch.zeros((B, H, nb), dtype=torch.float32, device=dev)
    bi = torch.zeros((B, H, nb, 2), dtype=torch.int16, device=dev)
    w = torch.tensor([weight], dtype=torch.float32, device=dev)
    err = lib().ref_self_collision_distance(_p(dist), _p(vec), _p(pd), _p(sparse), _p(spheres), _p(padding), _p(w),
                                            _p(pairs), _p(bv), _p(bi), nb, rm.max_threads_per_block, B, H, S,
                                            pairs.shape[0], 1, _stream(dev))
    assert err == 0, err
    return dist, vec


# ------------------------------------------------------------------------------------------------
# B-spline kernels of the reference (kernels/trajectory/bspline/bspline_kernel.cuh)
# ------------------------------------------------------------------------------------------------
def bspline_forward(knots, start, goal, start_idx, goal_idx, traj_dt, implicit, padded_horizon, degree):
    dev = knots.device
    B, nk, D = knots.shape
    outs = [torch.zeros((B, padded_horizon, D), dtype=torch.float32, device=dev) for _ in range(4)]
    odt = torch.zeros((B,), dtype=torch.float32, device=dev)
    err = lib().ref_bspline_forward(*[_p(o) for o in outs], _p(odt), _p(knots), *[_p(x) for x in start],
                                    *[_p(x) for x in goal], _p(start_idx), _p(goal_idx), _p(traj_dt), _p(implicit), B,
                                    padded_horizon, D, nk, degree, _stream(dev))
    assert err == 0, err
    return outs + [odt]


def bspline_single_dt(knots, start, goal, start_idx, goal_idx, interp_dt, implicit, interp_h, max_out_tsteps, degree):
    dev = knots.device
    B, nk, D = knots.shape
    outs = [torch.zeros((B, max_out_tsteps, D), dtype=torch.float32, device=dev) for _ in range(4)]
    odt = torch.zeros((B,), dtype=torch.float32, device=dev)
    err = lib().ref_bspline_single_dt(*[_p(o) for o in outs], _p(odt), _p(knots), None, *[_p(x) for x in start],
                                      *[_p(x) for x in goal], _p(start_idx), _p(goal_idx), _p(interp_dt), _p(implicit),
                                      _p(interp_h), B, max_out_tsteps, D, nk, degree, _stream(dev))
    assert err == 0, err
    return outs + [odt]


def bspline_backward(grads, traj_dt, dt_idx, implicit, n_knots, degree):
    dev = grads[0].device
    B, T, D = grads[0].shape
    out = torch.zeros((B, n_knots, D), dtype=torch.float32, device=dev)
    err = lib().ref_bspline_backward(_p(out), *[_p(g) for g in grads], _p(traj_dt), _p(dt_idx), _p(implicit), B, T, D,
                                     n_knots, degree, _stream(dev))
    assert err == 0, err
    return out


# ------------------------------------------------------------------------------------------------
# optimizer kernels of the reference (kernels/optimization/...): in-place on the passed tensors
# ------------------------------------------------------------------------------------------------
def lbfgs_step(step_vec, rho, y, s, q, x_0, grad_0, grad_q, epsilon, stable=True, use_shared=True):
    m, B, V = y.shape[0], y.shape[1], y.shape[2]
    err = lib().ref_lbfgs_step(_p(step_vec), _p(rho), _p(y), _p(s), _p(q), _p(x_0), _p(grad_0), _p(grad_q),
                               C.c_float(epsilon), B, m, V, int(stable), int(use_shared), _stream(y.device))
    assert err == 0, err
    return step_vec


def line_search(st, search_cost, search_action, search_gradient, step_direction, magnitudes, c_1, c_2, strong, approx,
                convergence_iteration=10, cost_delta_threshold=0.0, cost_relative_threshold=0.0):
    """st: dict of state tensors (best_cost, best_action, best_iteration, current_iteration, converged, exploration_*,
    selected_*, *_idx) updated in place."""
    B, n, V = search_action.shape
    err = lib().ref_line_search(
        _p(st["best_cost"]), _p(st["best_action"]), _p(st["best_iteration"]), _p(st["current_iteration"]), _p(st["converged"]),
        convergence_iteration, C.c_float(cost_delta_threshold), C.c_float(cost_relative_threshold),
        _p(st["exploration_cost"]), _p(st["exploration_action"]), _p(st["exploration_gradient"]), _p(st["exploration_idx"]),
        _p(st["selected_cost"]), _p(st["selected_action"]), _p(st["selected_gradient"]), _p(st["selected_idx"]),
        _p(search_cost), _p(search_action), _p(search_gradient), _p(step_direction), _p(magnitudes), C.c_float(c_1),
        C.c_float(c_2), int(strong), int(approx), n, V, B, _stream(search_cost.device))
    assert err == 0, err
    return st


# ------------------------------------------------------------------------------------------------
# RNEA kernels of the reference (kernels/dynamics/), serial path
# ------------------------------------------------------------------------------------------------
def rnea_forward(model, q, qd, qdd, nl, D, n_levels, out=None):
    """model = (fixed, mc, inertia, jtype, jmap, lmap, joff, gravity, level_starts, level_links) device tensors."""
    dev = q.device
    B = q.shape[0]
    if out is not None:
        tau, cache = out
    else:
        tau = torch.zeros((B, D), dtype=torch.float32, device=dev)
        cache = torch.zeros((B, nl * 20), dtype=torch.float32, device=dev)
    err = lib().ref_rnea_forward(_p(tau), _p(q), _p(qd), _p(qdd), *[_p(m) for m in model], _p(cache), B, nl, D, n_levels, _stream(dev))
    assert err == 0, err
    return tau, cache


def rnea_backward(model, grad_tau, q, qd, cache, nl, D, n_levels, out=None):
    dev = q.device
    B = q.shape[0]
    g = out if out is not None else [torch.zeros((B, D), dtype=torch.float32, device=dev) for _ in range(3)]
    err = lib().ref_rnea_backward(*[_p(x) for x in g], _p(grad_tau), _p(q), _p(qd), *[_p(m) for m in model], _p(cache), B, nl, D,
                                  n_levels, _stream(dev))
    assert err == 0, err
    return g


# ------------------------------------------------------------------------------------------------
# PBA+ 3-D EDT of the reference (kernels/parallel_banding/), its five launches + copy
# ------------------------------------------------------------------------------------------------
def pba3d(site_index, m3=2):
    """site_index [nx,ny,nz] int32 device tensor -> new tensor with the reference's nearest-site transform."""
    nx, ny, nz = site_index.shape
    out = site_index.contiguous().clone()
    buf = torch.empty_like(out)
    err = lib().ref_pba3d(_p(out), _p(buf), nx, ny, nz, m3, _stream(out.device))
    assert err == 0, err
    return out


# ------------------------------------------------------------------------------------------------
# FK with the centre of mass (COMPUTE_COM = true instantiations of the reference kernels)
# ------------------------------------------------------------------------------------------------
def fk_forward_com(kp, q, horizon=1):
    """q [N,D] -> (spheres, cumul, com [N,4]) through kinematics_forward_spheres_kernel<.., COMPUTE_COM=true>."""
    dev = q.device
    N = q.shape[0]
    z = lambda *s: torch.zeros(s, dtype=torch.float32, device=dev)  # noqa: E731
    pos, quat = z(N, kp.num_pose_links, 3), z(N, kp.num_pose_links, 4)
    sph, com, cum = z(N, kp.num_spheres, 4), z(N, 4), z(N, kp.num_links, 3, 4)
    eq = torch.zeros(1, dtype=torch.int32, device=dev)
    err = lib().ref_kinematics_forward_spheres_com(
        _p(pos), _p(quat), _p(sph), _p(com), _p(cum), _p(q), _p(kp.fixed_transforms), _p(kp.link_spheres),
        _p(kp.link_masses_com), _p(kp.joint_map_type), _p(kp.joint_map), _p(kp.link_map), _p(kp.tool_frame_map),
        _p(kp.link_sphere_idx_map), _p(kp.joint_offset_map), _p(eq), kp.num_envs, N, horizon, kp.num_dof,
        kp.num_spheres, kp.num_links, kp.num_pose_links, _stream(dev))
    assert err == 0, err
    return sph, cum, com


def fk_backward_com(kp, cumul, com, g_pos, g_quat, g_sph, g_com, horizon=1):
    dev = cumul.device
    N = cumul.shape[0]
    out = torch.zeros((N, kp.num_dof), dtype=torch.float32, device=dev)
    eq = torch.zeros(1, dtype=torch.int32, device=dev)
    err = lib().ref_kinematics_backward_com(
        _p(out), _p(g_pos), _p(g_quat), _p(g_sph), _p(g_com), _p(com), _p(cumul), _p(kp.link_spheres), _p(kp.link_masses_com),
        _p(kp.link_map), _p(kp.joint_map), _p(kp.joint_map_type), _p(kp.tool_frame_map), _p(kp.link_sphere_idx_map),
        _p(kp.link_chain_data), _p(kp.link_chain_offsets), _p(kp.joint_links_data), _p(kp.joint_links_offsets),
        _p(kp.joint_affects_endeffector), _p(kp.joint_offset_map), _p(eq), kp.num_envs, N, horizon, kp.num_dof, kp.num_spheres,
        kp.num_links, kp.num_pose_links, _stream(dev))
    assert err == 0, err
    return out
