"""GPU parity tests for hard / dynamic voxelization.  Everything here is bit-exact
(integer / byte work: coords, counts, order, point payloads)."""
import os

import numpy as np
import pytest
import torch

import oracle
from refgold import Gold

pytestmark = pytest.mark.gpu


def run_ours(cuda, pts, vs, cr, mp, mv):
    from bevfusion_b200.voxelize import voxelization
    v, c, n = voxelization(torch.from_numpy(pts).to(cuda), list(vs), list(cr), mp, mv, True)
    return v.cpu().numpy(), c.cpu().numpy(), n.cpu().numpy()


def assert_same(ours, gold):
    v, c, n = ours
    gv, gc, gn, gm = gold
    assert c.shape[0] == gm
    assert np.array_equal(c, gc), "voxel coords / order differ"
    assert np.array_equal(n, gn), "points-per-voxel differ"
    assert np.array_equal(v, gv), "voxel payloads differ"


@pytest.mark.parametrize("name", ["a", "b", "c"])
def test_golden_fixture(cuda, golden_dir, name):
    g = np.load(os.path.join(golden_dir, "voxelize_%s.npz" % name))
    ours = run_ours(cuda, g["points"], g["voxel_size"], g["coors_range"], int(g["max_points"]),
                    int(g["max_voxels"]))
    assert_same(ours, (g["voxels"], g["coors"], g["num_points"], int(g["voxel_num"])))


@pytest.mark.parametrize("n,mp,mv", [(1, 10, 5), (31, 2, 7), (4097, 10, 100000), (100000, 3, 3000)])
def test_random_noncubic_vs_oracle(cuda, n, mp, mv):
    from bevfusion_b200 import synthetic as S
    vs, cr = [0.4, 0.5, 0.25], [-8.0, -6.0, -1.0, 8.0, 6.0, 3.0]     # grid 40 x 24 x 16
    pts = S.uniform_cloud(n, seed=n, margin=1.0, rng_range=cr)
    assert_same(run_ours(cuda, pts, vs, cr, mp, mv), oracle.hard_voxelize(pts, vs, cr, mp, mv))


@pytest.mark.parametrize("shuffle", [True, False])
@pytest.mark.parametrize("max_voxels", [120000, 160000])
def test_full_size_c3(cuda, shuffle, max_voxels):
    """BASELINE config C3: ~296 k points, 0.075 m voxels, grid 1440x1440x40; both caps bind."""
    from bevfusion_b200 import synthetic as S
    pts = S.lidar_cloud(seed=0, shuffle=shuffle)
    L = S.LIDAR_C3
    gold = oracle.hard_voxelize(pts, L["voxel_size"], L["point_cloud_range"], 10, max_voxels)
    assert gold[3] == max_voxels                    # the synthetic cloud overflows the cap
    assert (gold[2] == 10).any()                    # and max_points binds
    assert_same(run_ours(cuda, pts, L["voxel_size"], L["point_cloud_range"], 10, max_voxels), gold)


def test_edge_cases(cuda):
    vs, cr = [0.5, 0.5, 0.5], [0, 0, 0, 4, 4, 2]
    v, c, n = run_ours(cuda, np.zeros((0, 4), np.float32), vs, cr, 3, 10)
    assert v.shape == (0, 3, 4) and c.shape == (0, 3) and n.shape == (0,)
    assert run_ours(cuda, np.full((100, 4), 100.0, np.float32), vs, cr, 3, 10)[1].shape[0] == 0
    # every point in ONE voxel (worst case for contention): first max_points indices survive
    pts = np.tile(np.array([[0.1, 0.1, 0.1, 0.0]], np.float32), (20000, 1))
    pts[:, 3] = np.arange(20000)
    assert_same(run_ours(cuda, pts, vs, cr, 7, 10), oracle.hard_voxelize(pts, vs, cr, 7, 10))
    # NaN / inf coordinates are dropped like out-of-range points
    pts = np.array([[0.1, 0.1, 0.1, 1], [np.nan, 0.1, 0.1, 2], [0.1, np.inf, 0.1, 3], [0.2, 0.2, 0.2, 4]],
                   np.float32)
    v, c, n = run_ours(cuda, pts, vs, cr, 3, 10)
    assert c.tolist() == [[0, 0, 0]] and n.tolist() == [2]


def test_dynamic_voxelize(cuda):
    from bevfusion_b200 import synthetic as S
    from bevfusion_b200.voxelize import voxelization
    vs, cr = [0.4, 0.5, 0.25], [-8.0, -6.0, -1.0, 8.0, 6.0, 3.0]
    pts = S.uniform_cloud(50000, seed=9, margin=1.0, rng_range=cr)
    coors = voxelization(torch.from_numpy(pts).to(cuda), vs, cr, -1, -1, True).cpu().numpy()
    assert np.array_equal(coors, oracle.dynamic_voxelize(pts, vs, cr))


def test_voxel_mean(cuda):
    from bevfusion_b200 import synthetic as S
    from bevfusion_b200.voxelize import voxelization, voxelize_mean
    vs, cr = [0.4, 0.5, 0.25], [-8.0, -6.0, -1.0, 8.0, 6.0, 3.0]
    pts = S.uniform_cloud(60000, seed=4, margin=0.5, rng_range=cr)
    v, c, n = voxelization(torch.from_numpy(pts).to(cuda), vs, cr, 10, 20000, True)
    feats, coords4 = voxelize_mean(v, c, n, batch_idx=3)
    gold = oracle.voxel_mean(v.cpu().numpy(), n.cpu().numpy())
    assert np.abs(feats.cpu().numpy() - gold).max() <= 1e-5 * np.abs(gold).max()
    assert torch.equal(coords4[:, 1:], c) and int(coords4[:, 0].min()) == 3 == int(coords4[:, 0].max())
    # and against the reference's torch expression (bevfusion.py:191-195)
    ref = v.sum(dim=1) / n.type_as(v).view(-1, 1)
    assert float((feats - ref).abs().max()) <= 1e-5 * float(ref.abs().max())


def reference_case_voxelize():
    """inputs of test_vs_reference_cuda_kernel: points, voxel size, range, max points, max voxels"""
    from bevfusion_b200 import synthetic as S
    L = S.LIDAR_C3
    pts = S.lidar_cloud(seed=1, sweeps=2)            # ~59 k points keeps the O(N^2) scan short
    return pts, L["voxel_size"], L["point_cloud_range"], 10, 20000


def test_vs_reference_cuda_kernel(cuda):
    """the reference's deterministic GPU voxelizer (O(N^2) + serial kernel), compiled unmodified."""
    gold = Gold("hard_voxelize")
    pts, vs, cr, mp, mv = reference_case_voxelize()
    assert int(gold["voxel_num"]) == mv
    v, c, n = run_ours(cuda, pts, vs, cr, mp, mv)
    assert c.shape[0] == mv
    gold.exact("coors", c)
    gold.exact("num_points", n)
    gold.exact("voxels", v)


def test_stress_c5_voxel_grid(cuda):
    """BASELINE config C5 LiDAR side: 0.05 m voxels -> grid 2160x2160x40; bit-exact vs the oracle,
    and the SubM / strided rulebooks on the 2160x2160x41 grid keep their invariants."""
    from bevfusion_b200 import synthetic as S
    from bevfusion_b200.spconv import ops
    from bevfusion_b200.voxelize import voxelize_mean
    pts = S.lidar_cloud(seed=2)
    vs, cr = [0.05, 0.05, 0.2], [-54.0, -54.0, -5.0, 54.0, 54.0, 3.0]
    gold = oracle.hard_voxelize(pts, vs, cr, 10, 300000)
    ours = run_ours(cuda, pts, vs, cr, 10, 300000)
    assert_same(ours, gold)
    v, c, n = (torch.from_numpy(a).to(cuda) for a in ours)
    feats, coords = voxelize_mean(v, c, n, 0)
    shape = [2160, 2160, 41]
    rb, _ = ops.get_rulebook(coords, 1, shape, 3, 1, 1, 1, 0, True)
    nbr = rb.nbr
    assert bool((nbr[13] == torch.arange(coords.shape[0], device=cuda, dtype=torch.int32)).all())   # centre tap = identity
    # SubM symmetry: j = nbr[k, i]  <=>  i = nbr[26 - k, j]
    k = 5
    i = torch.nonzero(nbr[k] >= 0).squeeze(1)
    j = nbr[k][i].long()
    assert bool((nbr[26 - k][j] == i.int()).all())
    rb2, oshape = ops.get_rulebook(coords, 1, shape, 3, 2, 1, 1, 0, False)
    assert oshape == [1080, 1080, 21]
    flat = oracle.flat_index(rb2.outids.cpu().numpy(), oshape)
    assert np.all(np.diff(flat) > 0)                         # ascending, unique output sites
    # every input feeds exactly one output through its parity-compatible offsets: pair count check
    pairs = int((rb2.nbr >= 0).sum())
    assert pairs >= coords.shape[0] and pairs <= 8 * coords.shape[0]


def test_voxelize_batch_matches_reference_glue(cuda):
    """voxelize_batch == the torch glue of BEVFusion.voxelize (bevfusion.py:169-197) on two samples."""
    import torch.nn.functional as F
    from bevfusion_b200 import synthetic as S
    from bevfusion_b200.voxelize import Voxelization, voxelize_batch
    vs, cr = [0.4, 0.5, 0.25], [-8.0, -6.0, -1.0, 8.0, 6.0, 3.0]
    pts = [torch.from_numpy(S.uniform_cloud(n, seed=n, margin=0.5, rng_range=cr)).to(cuda) for n in (30000, 17000)]
    vox = Voxelization(vs, cr, 10, (20000, 20000)).eval()
    feats, coords, sizes = voxelize_batch(pts, vox)
    rf, rc, rs = [], [], []
    for k, p in enumerate(pts):                                # the reference's loop, verbatim semantics
        f, c, n = vox(p)
        rf.append(f); rc.append(F.pad(c, (1, 0), mode="constant", value=k)); rs.append(n)
    rf, rc, rs = torch.cat(rf), torch.cat(rc), torch.cat(rs)
    rf = rf.sum(dim=1, keepdim=False) / rs.type_as(rf).view(-1, 1)
    assert torch.equal(coords, rc) and torch.equal(sizes, rs)
    assert float((feats - rf).abs().max()) <= 1e-5 * float(rf.abs().max())
    assert int(coords[:, 0].max()) == 1


def test_fused_voxelize_mean_full_size(cuda):
    """bevb200_hard_voxelize_mean == hard_voxelize followed by voxel_mean, at config C3 (caps bind),
    without the [M, 10, 5] intermediate: same voxel order, same counts, bit-identical means."""
    from bevfusion_b200 import synthetic as S
    from bevfusion_b200.voxelize import voxelization, voxelize_mean, voxelize_mean_fused
    L = S.LIDAR_C3
    pts = torch.from_numpy(S.lidar_cloud(seed=2)).to(cuda)
    for mv in (160000, 50000):
        v, c, n = voxelization(pts, L["voxel_size"], L["point_cloud_range"], 10, mv, True)
        feats, coords4 = voxelize_mean(v, c, n, batch_idx=1)
        f2, c2, n2 = voxelize_mean_fused(pts, L["voxel_size"], L["point_cloud_range"], 10, mv, batch_idx=1)
        assert f2.shape[0] == mv
        assert torch.equal(c2, coords4) and torch.equal(n2, n)
        assert torch.equal(f2, feats)
    # empty cloud
    f0, c0, n0 = voxelize_mean_fused(pts[:0], L["voxel_size"], L["point_cloud_range"], 10, 100)
    assert f0.shape == (0, 5) and c0.shape == (0, 4) and n0.shape == (0,)


def _scatter_case(n, ndim, seed, extent=12, neg_frac=0.1, c=5):
    rng = np.random.default_rng(seed)
    coors = rng.integers(0, extent, (n, ndim)).astype(np.int32)
    if ndim == 4:
        coors[:, 0] = np.sort(rng.integers(0, 3, n))            # batch column, grouped like the caller's
    bad = rng.random(n) < neg_frac
    coors[bad, rng.integers(1 if ndim == 4 else 0, ndim, bad.sum())] = -1
    feats = rng.standard_normal((n, c)).astype(np.float32)
    return feats, coors


@pytest.mark.parametrize("reduce_type", ["mean", "max", "sum"])
@pytest.mark.parametrize("n,ndim", [(1, 3), (257, 3), (20000, 3), (20000, 4), (300, 2)])
def test_dynamic_scatter_vs_oracle(cuda, reduce_type, n, ndim):
    from bevfusion_b200.voxelize import voxel_layer
    feats, coors = _scatter_case(n, ndim, seed=n + ndim)
    red, oc, cmap, cnt = voxel_layer.dynamic_point_to_voxel_forward(
        torch.from_numpy(feats).to(cuda), torch.from_numpy(coors).to(cuda), reduce_type)
    g_red, g_oc, g_map, g_cnt = oracle.dynamic_scatter(feats, coors, reduce_type)
    assert np.array_equal(oc.cpu().numpy(), g_oc)              # unique rows, lexicographic order
    assert np.array_equal(cmap.cpu().numpy(), g_map)
    assert np.array_equal(cnt.cpu().numpy(), g_cnt)
    if reduce_type == "max":
        assert np.array_equal(red.cpu().numpy(), g_red)
    else:
        assert np.abs(red.cpu().numpy() - g_red).max() <= 1e-5 * max(1.0, np.abs(g_red).max())
    # reproducible: same bits on a second run
    red2 = voxel_layer.dynamic_point_to_voxel_forward(
        torch.from_numpy(feats).to(cuda), torch.from_numpy(coors).to(cuda), reduce_type)[0]
    assert torch.equal(red, red2)


def test_dynamic_scatter_edge_cases(cuda):
    from bevfusion_b200.voxelize import voxel_layer
    # every row invalid -> no voxels, map all -1
    feats = torch.randn(10, 4, device=cuda)
    coors = torch.full((10, 3), -1, dtype=torch.int32, device=cuda)
    red, oc, cmap, cnt = voxel_layer.dynamic_point_to_voxel_forward(feats, coors, "mean")
    assert red.shape == (0, 4) and oc.shape == (0, 3) and cnt.shape == (0,)
    assert bool((cmap == -1).all())
    # no points
    red, oc, cmap, cnt = voxel_layer.dynamic_point_to_voxel_forward(feats[:0], coors[:0], "max")
    assert red.shape == (0, 4) and cmap.shape == (0,)
    # coordinates beyond the key range are an error, not silent aliasing
    big = torch.tensor([[0, 0, 1 << 20]], dtype=torch.int32, device=cuda)
    with pytest.raises(ValueError):
        voxel_layer.dynamic_point_to_voxel_forward(feats[:1], big, "sum")
    with pytest.raises(ValueError):
        voxel_layer.dynamic_point_to_voxel_forward(feats[:1], big, "median")


def reference_case_scatter(cuda):
    """inputs of test_dynamic_scatter_vs_reference_cuda_extension: LiDAR points and their voxel coordinates"""
    from bevfusion_b200 import synthetic as S
    from bevfusion_b200.voxelize import voxel_layer
    L = S.LIDAR_C3
    pts = torch.from_numpy(S.lidar_cloud(seed=3, sweeps=3)).to(cuda)
    coors = torch.zeros(pts.shape[0], 3, dtype=torch.int32, device=cuda)
    voxel_layer.dynamic_voxelize(pts, coors, L["voxel_size"], L["point_cloud_range"], 3)
    return pts, coors


def scatter_grad(red):
    return torch.randn(red.shape, generator=torch.Generator().manual_seed(red.shape[0])).to(red.device)


@pytest.mark.parametrize("reduce_type", ["mean", "max", "sum"])
def test_dynamic_scatter_vs_reference_cuda_extension(cuda, reduce_type):
    """forward and backward against the reference's own kernels (scatter_points_cuda.cu) compiled
    unmodified for sm_100, on the dynamic voxelization of a LiDAR cloud."""
    from bevfusion_b200.voxelize import voxel_layer
    gold = Gold("dynamic_scatter_" + reduce_type)
    pts, coors = reference_case_scatter(cuda)
    assert bool((coors < 0).any())                               # some points fall outside the range
    red, oc, cmap, cnt = voxel_layer.dynamic_point_to_voxel_forward(pts, coors, reduce_type)
    gold.exact("out_coors", oc)
    gold.exact("coors_map", cmap)
    gold.exact("count", cnt)
    if reduce_type == "max":
        gold.exact("reduced", red)
    else:
        gold.close("reduced", red, 1e-5)
    g = scatter_grad(red)
    grad = torch.full_like(pts, float("nan"))
    voxel_layer.dynamic_point_to_voxel_backward(grad, g, pts, red, cmap, cnt, reduce_type)
    if reduce_type == "max":
        gold.exact("grad", grad)
    else:
        gold.close("grad", grad, 1e-6)


@pytest.mark.parametrize("average", [True, False])
def test_dynamic_scatter_module_batched_autograd(cuda, average):
    """DynamicScatter on [N, 4] (batch, x, y, z) coors in one pass == the reference's per-sample
    python loop + cat (scatter_points.py:84-95); gradients match the oracle's backward."""
    from bevfusion_b200.scatter_points import DynamicScatter
    feats_np, coors_np = _scatter_case(5000, 4, seed=9, extent=9)
    feats = torch.from_numpy(feats_np).to(cuda).requires_grad_(True)
    coors = torch.from_numpy(coors_np).to(cuda)
    mod = DynamicScatter([0.1, 0.1, 0.1], [0, 0, 0, 1, 1, 1], average)
    vf, vc = mod(feats, coors)
    reduce_type = "mean" if average else "max"
    gf, gc = [], []
    for b in range(int(coors_np[-1, 0]) + 1):                   # the reference's loop
        sel = coors_np[:, 0] == b
        r, oc, _, _ = oracle.dynamic_scatter(feats_np[sel], coors_np[sel][:, 1:], reduce_type)
        gf.append(r); gc.append(np.pad(oc, ((0, 0), (1, 0)), constant_values=b))
    gf, gc = np.concatenate(gf), np.concatenate(gc)
    assert np.array_equal(vc.cpu().numpy(), gc)
    assert np.abs(vf.detach().cpu().numpy() - gf).max() <= 1e-5 * np.abs(gf).max()
    w = torch.randn_like(vf)
    (vf * w).sum().backward()
    red, oc, cmap, cnt = oracle.dynamic_scatter(feats_np, coors_np, reduce_type)
    gold = oracle.dynamic_scatter_backward(w.cpu().numpy(), feats_np, red, cmap, cnt, reduce_type)
    assert np.abs(feats.grad.cpu().numpy() - gold).max() <= 1e-6 * max(1.0, np.abs(gold).max())
