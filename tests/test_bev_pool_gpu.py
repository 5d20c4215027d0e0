"""GPU parity tests for bev_pool: CUDA path (through the C ABI) vs the CPU oracle, the committed
golden fixture, and the stored outputs of the reference's own CUDA kernels (tests/refgold.py).
Tolerances: ranks / perm / interval tables bit-exact; pooled features <= 1e-4 relative
(BASELINE.json north_star); backward is a pure copy -> bit-exact."""
import os

import numpy as np
import pytest
import torch

import oracle
from refgold import Gold

pytestmark = pytest.mark.gpu


def rel_err(got, gold):
    return float(np.abs(got.astype(np.float64) - gold.astype(np.float64)).max() / max(np.abs(gold).max(), 1e-30))


def random_case(n, c, B, D, H, W, seed, hot_cells=0):
    rng = np.random.default_rng(seed)
    coords = np.stack([rng.integers(0, H, n), rng.integers(0, W, n), rng.integers(0, D, n),
                       rng.integers(0, B, n)], 1).astype(np.int64)
    if hot_cells:  # a few cells that collect very long intervals (> 2 chunks)
        hot = rng.integers(0, n, size=n // 3)
        coords[hot] = coords[rng.integers(0, n, hot_cells)][rng.integers(0, hot_cells, hot.size)]
    feats = rng.standard_normal((n, c)).astype(np.float32)
    return feats, coords


def sorted_inputs(feats, coords, B, D, H, W):
    ranks = oracle.ranks_of(coords, B, D, H, W)
    order, rs, starts, lengths = oracle.sort_and_intervals(ranks)
    return feats[order], coords[order].astype(np.int32), rs, starts, lengths, order


@pytest.mark.parametrize("c", [80, 64, 128, 16, 32, 96, 160, 256, 20, 7])
def test_forward_ext_vs_oracle(cuda, c):
    from bevfusion_b200.bev_pool import bev_pool_ext
    B, D, H, W = 2, 2, 24, 20
    feats, coords = random_case(30000, c, B, D, H, W, seed=c, hot_cells=3)
    x, g, rs, starts, lengths, _ = sorted_inputs(feats, coords, B, D, H, W)
    assert lengths.max() > 600          # exercises the long-interval (multi-chunk) path
    gold = oracle.bev_pool_forward(x, g, lengths, starts, B, D, H, W, acc64=True)
    out = bev_pool_ext.bev_pool_forward(torch.from_numpy(x).to(cuda), torch.from_numpy(g).to(cuda),
                                        torch.from_numpy(lengths).to(cuda),
                                        torch.from_numpy(starts).to(cuda), B, D, H, W)
    assert tuple(out.shape) == (B, D, H, W, c)
    assert rel_err(out.cpu().numpy(), gold) <= 1e-4
    # run-to-run bit reproducibility (no float atomics)
    out2 = bev_pool_ext.bev_pool_forward(torch.from_numpy(x).to(cuda), torch.from_numpy(g).to(cuda),
                                         torch.from_numpy(lengths).to(cuda),
                                         torch.from_numpy(starts).to(cuda), B, D, H, W)
    assert torch.equal(out, out2)


def test_backward_ext_vs_oracle_bit_exact(cuda):
    from bevfusion_b200.bev_pool import bev_pool_ext
    B, D, H, W, c = 2, 1, 16, 12, 80
    feats, coords = random_case(9000, c, B, D, H, W, seed=11, hot_cells=2)
    x, g, rs, starts, lengths, _ = sorted_inputs(feats, coords, B, D, H, W)
    og = np.random.default_rng(1).standard_normal((B, D, H, W, c)).astype(np.float32)
    gold = oracle.bev_pool_backward(og, g, lengths, starts, B, D, H, W)
    got = bev_pool_ext.bev_pool_backward(torch.from_numpy(og).to(cuda), torch.from_numpy(g).to(cuda),
                                         torch.from_numpy(lengths).to(cuda),
                                         torch.from_numpy(starts).to(cuda), B, D, H, W)
    assert np.array_equal(got.cpu().numpy(), gold)


def test_tables_bit_exact_vs_oracle(cuda):
    """rank / stable sort / interval table computed by the library == oracle (bit-exact)."""
    from bevfusion_b200.bev_pool import prepare_from_coords
    B, D, H, W = 3, 2, 40, 33
    _, coords = random_case(50000, 4, B, D, H, W, seed=5, hot_cells=2)
    t = prepare_from_coords(torch.from_numpy(coords).to(cuda), B, D, H, W)
    ranks = oracle.ranks_of(coords, B, D, H, W)
    order, rs, starts, lengths = oracle.sort_and_intervals(ranks)
    assert t.n_kept == coords.shape[0] and t.n_intervals == starts.shape[0]
    assert np.array_equal(t.ranks[:t.n_kept].cpu().numpy(), rs.astype(np.int32))
    assert np.array_equal(t.perm[:t.n_kept].cpu().numpy(), order.astype(np.int32))   # stable
    assert np.array_equal(t.geom.cpu().numpy(), coords[order].astype(np.int32))
    assert np.array_equal(t.starts.cpu().numpy(), starts)
    assert np.array_equal(t.lengths.cpu().numpy(), lengths)


def test_geometry_quantise_filter_bit_exact(cuda):
    """quantise + filter + rank from fp32 geometry (base.py:149-169) is bit-exact."""
    from bevfusion_b200 import synthetic as S
    from bevfusion_b200.bev_pool import gen_dx_bx, prepare_from_geometry
    geom, cfg = S.camera_geometry("tiny", batch=2)
    g = geom.clone()
    g.view(-1, 3)[:200, 0] = -16.0 - 1e-4        # in (-1, 0): truncates to cell 0 and is KEPT
    g.view(-1, 3)[200:300, 1] = 16.0             # exactly on the upper bound: dropped
    dx, bx, nx = gen_dx_bx(cfg["xbound"], cfg["ybound"], cfg["zbound"])
    t = prepare_from_geometry(g.to(cuda), dx, bx, nx, 2)
    odx, obx, onx = oracle.gen_dx_bx(cfg["xbound"], cfg["ybound"], cfg["zbound"])
    coords, kept = oracle.quantize_filter(g.numpy(), odx, obx, onx, 2)
    ranks = oracle.ranks_of(coords[kept], 2, int(onx[2]), int(onx[0]), int(onx[1]))
    order, rs, starts, lengths = oracle.sort_and_intervals(ranks)
    kept_idx = np.nonzero(kept)[0]
    assert t.n_kept == int(kept.sum()) and t.n_intervals == starts.shape[0]
    assert np.array_equal(t.ranks[:t.n_kept].cpu().numpy(), rs.astype(np.int32))
    assert np.array_equal(t.perm[:t.n_kept].cpu().numpy(), kept_idx[order].astype(np.int32))
    assert np.array_equal(np.sort(t.perm[t.n_kept:].cpu().numpy()), np.nonzero(~kept)[0])
    assert np.array_equal(t.starts.cpu().numpy(), starts)
    assert np.array_equal(t.lengths.cpu().numpy(), lengths)
    assert np.array_equal(t.geom.cpu().numpy(), coords[kept][order].astype(np.int32))


def test_drop_in_bev_pool_forward_backward(cuda):
    """bev_pool(feats, coords, B, D, H, W) -> [B, C, D, H, W]; autograd gives grads in the
    caller's row order."""
    from bevfusion_b200.bev_pool import bev_pool
    B, D, H, W, c = 2, 2, 12, 10, 16
    feats, coords = random_case(6000, c, B, D, H, W, seed=3)
    gold = oracle.bev_pool(feats, coords, B, D, H, W)
    x = torch.from_numpy(feats).to(cuda).requires_grad_(True)
    out = bev_pool(x, torch.from_numpy(coords).to(cuda), B, D, H, W)
    assert tuple(out.shape) == (B, c, D, H, W)
    assert rel_err(out.detach().cpu().numpy(), gold) <= 1e-4
    w = torch.randn_like(out)
    (out * w).sum().backward()
    wn = w.cpu().numpy()
    gold_grad = wn[coords[:, 3], :, coords[:, 2], coords[:, 0], coords[:, 1]]
    assert np.array_equal(x.grad.cpu().numpy(), gold_grad)


def test_golden_fixture(cuda, golden_dir):
    """the committed reference-QuickCumsum fixture (tests/golden/make_golden.py)."""
    from bevfusion_b200.bev_pool import bev_pool
    g = np.load(os.path.join(golden_dir, "bev_pool_quickcumsum.npz"))
    B, D, H, W = (int(v) for v in g["dims"])
    out = bev_pool(torch.from_numpy(g["feats"]).to(cuda), torch.from_numpy(g["coords"]).to(cuda),
                   B, D, H, W).cpu().numpy()
    pg = g["pooled_geom"]
    got = out[pg[:, 3], :, pg[:, 2], pg[:, 0], pg[:, 1]]
    assert np.abs(got - g["pooled"]).max() < 5e-4       # QuickCumsum's own cancellation error


def test_empty_and_single(cuda):
    from bevfusion_b200.bev_pool import bev_pool, bev_pool_ext
    z = bev_pool_ext.bev_pool_forward(torch.zeros(0, 80, device=cuda),
                                      torch.zeros(0, 4, dtype=torch.int32, device=cuda),
                                      torch.zeros(0, dtype=torch.int32, device=cuda),
                                      torch.zeros(0, dtype=torch.int32, device=cuda), 1, 1, 4, 4)
    assert float(z.abs().sum()) == 0 and tuple(z.shape) == (1, 1, 4, 4, 80)
    out = bev_pool(torch.ones(1, 80, device=cuda), torch.tensor([[3, 2, 0, 0]], device=cuda), 1, 1, 4, 4)
    assert float(out.sum()) == 80 and float(out[0, :, 0, 3, 2].sum()) == 80


def reference_case_kernel(cuda):
    """inputs of test_vs_reference_cuda_kernel: sorted rows, tables, dims and an output gradient"""
    B, D, H, W, c = 1, 1, 64, 64, 80
    feats, coords = random_case(200000, c, B, D, H, W, seed=21, hot_cells=4)
    x, g, rs, starts, lengths, _ = sorted_inputs(feats, coords, B, D, H, W)
    args = [torch.from_numpy(a).to(cuda) for a in (x, g, lengths, starts)]
    og = torch.randn((B, D, H, W, c), generator=torch.Generator().manual_seed(22)).to(cuda)
    return args, (B, D, H, W), og


def test_vs_reference_cuda_kernel(cuda):
    """the reference's own bev_pool CUDA kernels, compiled unmodified for sm_100."""
    from bevfusion_b200.bev_pool import bev_pool_ext
    gold = Gold("bev_pool_kernel")
    args, dims, og = reference_case_kernel(cuda)
    out = bev_pool_ext.bev_pool_forward(*args, *dims)
    gold.close("forward", out, 1e-4)
    got_g = bev_pool_ext.bev_pool_backward(og, args[1], args[2], args[3], *dims)
    gold.exact("backward", got_g)


def test_plan_full_size_c2_properties(cuda):
    """BASELINE config C2 (6 cam, 32x88 features, D=118, C=80, 360x360): plan path vs a float64
    torch index_add_ gold on the device, plus size-independent properties (mass conservation,
    linearity) and reference-path equivalence."""
    from bevfusion_b200 import synthetic as S
    from bevfusion_b200.bev_pool import BEVPoolPlan
    geom, cfg = S.camera_geometry("C2", device=cuda)
    plan = BEVPoolPlan(geom, cfg["xbound"], cfg["ybound"], cfg["zbound"])
    t = plan.tables
    assert t.n_total == 6 * 118 * 32 * 88
    x = S.lifted_features("C2", device=cuda, seed=0)
    out = plan.pool(x)                                    # [1, 1, 360, 360, 80]
    xf = x.reshape(-1, 80)
    perm = t.perm[:t.n_kept].long()
    # gold: float64 scatter-add by cell on the device
    cell = (t.geom[:, 0].long() * 360 + t.geom[:, 1].long())
    gold = torch.zeros(360 * 360, 80, dtype=torch.float64, device=cuda)
    gold.index_add_(0, cell, xf[perm].double())
    err = (out.reshape(-1, 80).double() - gold).abs().max() / gold.abs().max()
    assert float(err) <= 1e-4
    # mass conservation: sum of the grid == sum of the kept rows
    assert abs(float(out.double().sum() - xf[perm].double().sum())) <= 1e-6 * float(xf[perm].double().abs().sum())
    # linearity: pool(2x) == 2 pool(x) exactly (power-of-two scaling is exact in fp32)
    assert torch.equal(plan.pool(x * 2.0), out * 2.0)
    # layout of the module-level call == BaseTransform.bev_pool
    bev = plan(x)
    assert tuple(bev.shape) == (1, 80, 360, 360)
    assert torch.equal(bev[0, :, 17, 200], out[0, 0, 17, 200, :])
    # backward: grad of sum(out * w) w.r.t. x is w[cell] for kept rows, 0 for dropped rows
    xg = x.clone().requires_grad_(True)
    w = torch.randn_like(out)
    (plan.pool(xg) * w).sum().backward()
    gflat = xg.grad.reshape(-1, 80)
    assert torch.equal(gflat[perm], w.reshape(-1, 80)[cell])
    dropped = t.perm[t.n_kept:].long()
    assert float(gflat[dropped].abs().sum()) == 0.0


def reference_case_c2(cuda):
    """inputs of test_plan_full_size_c2_vs_reference_cuda_kernel: the C2 plan and a lifted volume"""
    from bevfusion_b200 import synthetic as S
    from bevfusion_b200.bev_pool import BEVPoolPlan
    geom, cfg = S.camera_geometry("C2", device=cuda)
    plan = BEVPoolPlan(geom, cfg["xbound"], cfg["ybound"], cfg["zbound"])
    return plan, S.lifted_features("C2", device=cuda, seed=1)


def test_plan_full_size_c2_vs_reference_cuda_kernel(cuda):
    """BASELINE config C2 against the reference's OWN CUDA kernel (compiled unmodified for sm_100): the reference
    path materialises x[perm] (592 MB) and runs bev_pool_forward on the sorted rows with the interval tables; the plan
    path pools the unsorted volume through perm.  Same cells, same rows per cell in the same order -> <= 1e-4 (in fact
    equal up to the summation tree of the wide intervals)."""
    gold = Gold("bev_pool_c2")
    plan, x = reference_case_c2(cuda)
    out = plan.pool(x)                                               # [1, 1, 360, 360, 80]
    gold.close("forward", out, 1e-4)
    gold.exact("nonzero", out != 0)


@pytest.mark.parametrize("cfg_name", ["tiny", "C2"])
def test_fused_lift_pool(cuda, cfg_name):
    """fused LSS lift + pool == pool(depth (x) ctx) without the materialised volume."""
    from bevfusion_b200 import synthetic as S
    from bevfusion_b200.bev_pool import BEVPoolPlan
    geom, cfg = S.camera_geometry(cfg_name, device=cuda)
    plan = BEVPoolPlan(geom, cfg["xbound"], cfg["ybound"], cfg["zbound"])
    B, N, D, fH, fW, _ = geom.shape
    C = cfg["C"]
    g = torch.Generator(device=cuda).manual_seed(1)
    depth = torch.softmax(torch.randn(B, N, D, fH, fW, generator=g, device=cuda), dim=2).contiguous()
    ctx = torch.randn(B, N, fH, fW, C, generator=g, device=cuda)
    x = depth.unsqueeze(-1) * ctx.unsqueeze(2)                  # [B, N, D, fH, fW, C]  (the reference's lift)
    gold = plan.pool(x)
    out = plan.lift_pool(depth, ctx)
    scale = float(gold.abs().max())
    # the column kernel adds the same fp32 products in a different (fixed) order than the row-wise pooling
    assert float((out - gold).abs().max()) <= 1e-5 * scale
    assert bool(torch.equal(out, plan.lift_pool(depth, ctx)))               # reproducible
    assert bool(((out != 0).any(-1) == (gold != 0).any(-1)).all())          # same occupied cells, zero elsewhere
    os.environ["BEVB200_LIFT_VARIANT"] = "rows"                             # round-1 kernel: same order as pool()
    try:
        rows = plan.lift_pool(depth, ctx)
    finally:
        del os.environ["BEVB200_LIFT_VARIANT"]
    assert float((rows - gold).abs().max()) <= 1e-6 * scale
    # and against a float64 scatter-add of the lifted volume
    t = plan.tables
    perm = t.perm[:t.n_kept].long()
    nxy = int(plan.nx[0]) * int(plan.nx[1])
    cell = t.geom[:, 0].long() * int(plan.nx[1]) + t.geom[:, 1].long()
    ref = torch.zeros(nxy, C, dtype=torch.float64, device=cuda)
    ref.index_add_(0, cell, x.reshape(-1, C)[perm].double())
    assert float((out.reshape(-1, C).double() - ref).abs().max()) <= 1e-4 * float(ref.abs().max())


@pytest.mark.parametrize("batch", [1, 2])
def test_fused_lift_pool_arbitrary_geometry(cuda, batch):
    """the column lift assumes nothing about the cameras: with frustum points jittered so that the pixels of an
    image column scatter over many cells (and some leave the grid), every (column, depth, cell) group still
    becomes its own segment and the result equals pooling the materialised volume.  batch 2: no zero-fill
    shortcut (cells are not ascending in interval order)."""
    from bevfusion_b200 import synthetic as S
    from bevfusion_b200.bev_pool import BEVPoolPlan
    geom, cfg = S.camera_geometry("tiny", batch=batch, device=cuda)
    g = torch.Generator(device=cuda).manual_seed(7)
    geom = geom + torch.randn(geom.shape, generator=g, device=cuda) * 1.5      # metres: several cells
    plan = BEVPoolPlan(geom.contiguous(), cfg["xbound"], cfg["ybound"], cfg["zbound"])
    B, N, D, fH, fW, _ = geom.shape
    C = 64
    depth = torch.softmax(torch.randn(B, N, D, fH, fW, generator=g, device=cuda), dim=2).contiguous()
    ctx = torch.randn(B, N, fH, fW, C, generator=g, device=cuda)
    gold = plan.pool(depth.unsqueeze(-1) * ctx.unsqueeze(2))
    out = plan.lift_pool(depth, ctx)
    assert float((out - gold).abs().max()) <= 1e-5 * float(gold.abs().max())
    n_seg = plan._lift_cache[1][5]
    assert plan.tables.n_intervals <= n_seg <= plan.tables.n_kept
    assert n_seg > 0.5 * plan.tables.n_kept                                    # most jittered points sit alone in their segment


@pytest.mark.parametrize("cfg_name,batch", [("tiny", 2), ("C2", 1)])
def test_plan_from_cameras_matches_torch_geometry(cuda, cfg_name, batch):
    """get_geometry fused into the plan build (explicit fp32, fixed summation order) against torch's get_geometry
    followed by the plan build: the geometry agrees to fp32 rounding, and the tables are identical except for the
    handful of frustum points that sit within rounding of a cell boundary (each off by one cell)."""
    from bevfusion_b200 import synthetic as S
    from bevfusion_b200.bev_pool import BEVPoolPlan, gen_dx_bx, prepare_from_cameras
    from bevfusion_b200.vtransform import create_frustum, get_geometry
    cfg = S.CONFIGS[cfg_name]
    rig = {k: v.to(cuda) for k, v in S.camera_rig(cfg["n_cam"], cfg["image_size"], batch).items()}
    extra_r = extra_t = None
    if batch > 1:                                           # a lidar augmentation per sample
        M = S.lidar_camera_matrices(cfg["n_cam"], cfg["image_size"], batch)["lidar_aug_matrix"].to(cuda)
        extra_r, extra_t = M[:, :3, :3].contiguous(), M[:, :3, 3].contiguous()
    frustum = create_frustum(cfg["image_size"], cfg["feature_size"], cfg["dbound"]).to(cuda)
    geom = get_geometry(frustum, rig["camera2lidar_rots"], rig["camera2lidar_trans"], rig["intrins"],
                        rig["post_rots"], rig["post_trans"], extra_r, extra_t).contiguous()
    ref = BEVPoolPlan(geom, cfg["xbound"], cfg["ybound"], cfg["zbound"])
    dx, bx, nx = gen_dx_bx(cfg["xbound"], cfg["ybound"], cfg["zbound"])
    tabs, g2 = prepare_from_cameras(frustum, rig["camera2lidar_rots"], rig["camera2lidar_trans"], rig["intrins"],
                                    rig["post_rots"], rig["post_trans"], dx, bx, nx, extra_r, extra_t,
                                    return_geometry=True)
    g1 = geom.reshape(-1, 3)
    assert float((g1 - g2).abs().max()) <= 2e-5 * float(g1.abs().max())
    n = g1.shape[0]
    rank_ref = torch.full((n,), -1, dtype=torch.int64, device=cuda)
    rank_ref[ref.tables.perm[:ref.tables.n_kept].long()] = ref.tables.ranks[:ref.tables.n_kept].long()
    rank_new = torch.full((n,), -1, dtype=torch.int64, device=cuda)
    rank_new[tabs.perm[:tabs.n_kept].long()] = tabs.ranks[:tabs.n_kept].long()
    differ = rank_ref != rank_new
    assert float(differ.float().mean()) <= 2e-4                 # boundary points only
    # every differing point is within rounding of a cell boundary in at least one axis
    if bool(differ.any()):
        lower = (bx - dx / 2.0).to(cuda)
        frac = ((g1[differ] - lower) / dx.to(cuda))
        dist = (frac - frac.round()).abs().min(dim=1).values
        assert float(dist.max()) <= 1e-3
    plan = BEVPoolPlan.from_cameras(frustum, rig["camera2lidar_rots"], rig["camera2lidar_trans"], rig["intrins"],
                                    rig["post_rots"], rig["post_trans"], cfg["xbound"], cfg["ybound"], cfg["zbound"],
                                    extra_r, extra_t)
    assert plan.tables.n_kept == tabs.n_kept and bool(torch.equal(plan.tables.perm, tabs.perm))
    assert abs(plan.tables.n_kept - ref.tables.n_kept) <= max(4, int(2e-4 * n))


def test_stress_c5_properties(cuda):
    """BASELINE config C5 (6 cam 512x1408 -> 64x176 features, D=200, C=80, 256x256 BEV:
    N' = 13.5 M rows, x = 4.3 GB): size-independent properties of the plan path at full size."""
    from bevfusion_b200 import synthetic as S
    from bevfusion_b200.bev_pool import BEVPoolPlan
    geom, cfg = S.camera_geometry("C5", device=cuda)
    assert geom.shape[2] == 200 or geom.shape[2] == len(np.arange(*cfg["dbound"]))
    plan = BEVPoolPlan(geom, cfg["xbound"], cfg["ybound"], cfg["zbound"])
    t = plan.tables
    n_total = geom.numel() // 3
    assert t.n_total == n_total
    del geom
    # table invariants: perm is a permutation, intervals tile [0, n_kept), ranks ascend strictly per interval
    perm = t.perm.long()
    seen = torch.zeros(n_total, dtype=torch.bool, device=cuda)
    seen[perm] = True
    assert bool(seen.all())
    assert int(t.lengths.sum()) == t.n_kept and int(t.starts[0]) == 0
    assert bool((t.starts[1:] - t.starts[:-1] == t.lengths[:-1]).all())
    rk = t.ranks[:t.n_kept]
    assert bool((rk[1:] >= rk[:-1]).all())
    assert bool((rk[t.starts[1:].long()] > rk[t.starts[1:].long() - 1]).all())
    # pooling a volume of ones counts the points of every cell (exact in fp32: counts < 2^24)
    C = 80
    x = torch.ones((n_total, C), device=cuda)
    out = plan.pool(x)                                        # [1, 1, 256, 256, 80]
    counts = torch.zeros(256 * 256, dtype=torch.float32, device=cuda)
    cell = t.geom[:, 0].long() * 256 + t.geom[:, 1].long()
    counts.index_add_(0, cell[t.starts.long()], t.lengths.float())
    assert torch.equal(out.reshape(-1, C)[:, 0], counts) and torch.equal(out.reshape(-1, C)[:, 79], counts)
    assert int(t.lengths.max()) > 1000                       # very long intervals exist at this size
    # mass conservation on random data
    x.normal_()
    out = plan.pool(x)
    kept_sum = x[perm[:t.n_kept]].double().sum()
    assert abs(float(out.double().sum() - kept_sum)) <= 1e-6 * float(x[perm[:t.n_kept]].double().abs().sum())


def test_prepare_vs_reference_vtransform_fixture(cuda, golden_dir):
    """device precompute (quantise / filter / rank / sort) vs the coords the REFERENCE's
    BaseTransform.bev_pool produced for the same geometry (fixture from the reference source)."""
    from bevfusion_b200.bev_pool import gen_dx_bx, prepare_from_geometry
    from bevfusion_b200 import synthetic as S
    g = np.load(os.path.join(golden_dir, "vtransform_tiny.npz"))
    cfg = S.CONFIGS["tiny"]
    dx, bx, nx = gen_dx_bx(cfg["xbound"], cfg["ybound"], cfg["zbound"])
    t = prepare_from_geometry(torch.from_numpy(g["geom"]).to(cuda), dx, bx, nx, 2)
    B, D, H, W = (int(v) for v in g["dims"])
    ref_coords = g["coords"]                                       # kept rows, original order
    assert t.n_kept == ref_coords.shape[0]
    ranks = oracle.ranks_of(ref_coords, B, D, H, W)
    order, rs, starts, lengths = oracle.sort_and_intervals(ranks)
    assert np.array_equal(t.ranks[:t.n_kept].cpu().numpy(), rs.astype(np.int32))
    assert np.array_equal(t.geom.cpu().numpy(), ref_coords[order].astype(np.int32))
    assert np.array_equal(t.starts.cpu().numpy(), starts) and np.array_equal(t.lengths.cpu().numpy(), lengths)


def test_plan_layout_matches_reference_path_multi_z(cuda):
    """plan(x) == BaseTransform.bev_pool(geom, x) (torch index glue + drop-in op + permute + cat)
    on a grid with B = 2 samples and nz = 2 height bins."""
    from bevfusion_b200 import synthetic as S
    from bevfusion_b200.bev_pool import BEVPoolPlan
    from bevfusion_b200.vtransform import LSSGeometry
    cfg = dict(S.CONFIGS["tiny"]); cfg["zbound"] = (-10.0, 10.0, 10.0)
    geom, _ = S.camera_geometry("tiny", batch=2, device=cuda)
    lss = LSSGeometry(cfg["image_size"], cfg["feature_size"], cfg["xbound"], cfg["ybound"], cfg["zbound"],
                      cfg["dbound"]).to(cuda)
    x = S.lifted_features("tiny", batch=2, device=cuda, seed=3)
    ref = lss.bev_pool_reference_path(geom, x)                  # [2, 80*2, 64, 64]
    plan = BEVPoolPlan(geom, cfg["xbound"], cfg["ybound"], cfg["zbound"])
    out = plan(x)
    assert tuple(out.shape) == tuple(ref.shape) == (2, 160, 64, 64)
    assert float((out - ref).abs().max()) <= 1e-5 * float(ref.abs().max())


def test_fuser_input_written_in_place(cuda):
    """camera BEV (plan output) and LiDAR BEV (encoder dense output) written straight into the
    channel slices of one [B, 80+256, X, Y] buffer == torch.cat of the separate results
    (fusers/conv.py:16)."""
    from bevfusion_b200 import synthetic as S
    from bevfusion_b200.bev_pool import BEVPoolPlan
    from bevfusion_b200.spconv import ops as sp_ops
    cfg = dict(S.CONFIGS["tiny"]); cfg["zbound"] = (-10.0, 10.0, 10.0)
    geom, _ = S.camera_geometry("tiny", batch=2, device=cuda)
    x = S.lifted_features("tiny", batch=2, device=cuda, seed=3)
    plan = BEVPoolPlan(geom, cfg["xbound"], cfg["ybound"], cfg["zbound"])
    cam = plan(x)
    B, CC, X, Y = cam.shape
    rng = np.random.default_rng(0)
    n, c, Z = 500, 8, 2
    idx = np.unique(np.stack([rng.integers(0, B, n), rng.integers(0, X, n), rng.integers(0, Y, n),
                              rng.integers(0, Z, n)], 1), axis=0).astype(np.int32)
    feats = torch.from_numpy(rng.standard_normal((idx.shape[0], c)).astype(np.float32)).to(cuda)
    indices = torch.from_numpy(idx).to(cuda)
    lidar = sp_ops.sparse_to_dense(feats, indices, B, (X, Y, Z), z_major=True)
    buf = torch.full((B, CC + c * Z, X, Y), float("nan"), device=cuda)
    plan(x, out=buf[:, :CC])
    sp_ops.sparse_to_dense(feats, indices, B, (X, Y, Z), z_major=True, out=buf[:, CC:])
    assert torch.equal(buf, torch.cat([cam, lidar], 1))
    with pytest.raises(ValueError):
        plan(x, out=buf[:, :, :, 1:])
