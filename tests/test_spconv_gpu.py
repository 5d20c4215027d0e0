"""GPU parity tests for the sparse-conv path: rulebook (bit-exact as index sets / output order),
implicit-GEMM conv and the SparseEncoder (<= 1e-4 relative, BASELINE.json north_star) against
the CPU oracle, the committed reference fixtures and the stored outputs of the reference's CUDA extension."""
import glob
import os

import numpy as np
import pytest
import torch

import oracle
from refgold import Gold

pytestmark = pytest.mark.gpu

PRECISIONS = [0]  # BEVB200_PREC_FP32; tensor-core modes are appended when built
if os.environ.get("BEVB200_TEST_TC", "1") == "1":
    PRECISIONS += [1]


def tc_available(cuda):
    """True when the tcgen05 path is compiled in (the placeholder returns EUNSUPPORTED)."""
    from bevfusion_b200.spconv import ops
    from bevfusion_b200._C import BevB200Error
    try:
        f = torch.zeros(4, 16, device=cuda)
        w = torch.zeros(1, 16, 16, device=cuda)
        nbr = torch.zeros(1, 4, dtype=torch.int32, device=cuda)
        ops.sparse_conv(f, w, nbr, 4, precision=1)
        return True
    except BevB200Error:
        return False


def rel_err(got, gold):
    return float(np.abs(got.astype(np.float64) - gold.astype(np.float64)).max() / max(np.abs(gold).max(), 1e-30))


def random_sparse(n, shape, B, seed):
    rng = np.random.default_rng(seed)
    vol = B * shape[0] * shape[1] * shape[2]
    flat = rng.choice(vol, size=n, replace=False)
    z = flat % shape[2]; y = (flat // shape[2]) % shape[1]
    x = (flat // (shape[2] * shape[1])) % shape[0]; b = flat // (shape[2] * shape[1] * shape[0])
    return np.stack([b, x, y, z], 1).astype(np.int32)


def pair_table(pairs, num):
    """a rulebook as one canonical array: (offset, in, out) rows in ascending order"""
    p, n = pairs.cpu().numpy(), num.cpu().numpy()
    t = np.concatenate([np.stack([np.full(n[k], k), p[k, 0, :n[k]], p[k, 1, :n[k]]], 1)
                        for k in range(p.shape[0])]).astype(np.int64)
    return t[np.lexsort(t.T[::-1])]


def out_grad(n, c, seed):
    return torch.randn((n, c), generator=torch.Generator().manual_seed(seed))


def pair_sets(pairs, num):
    return [set(zip(pairs[k, 0, :num[k]].tolist(), pairs[k, 1, :num[k]].tolist()))
            for k in range(pairs.shape[0])]


GEOMS = {
    "subm_k3": ([3, 3, 3], [1, 1, 1], [1, 1, 1], True),
    "conv_k3s2p1": ([3, 3, 3], [2, 2, 2], [1, 1, 1], False),
    "conv_k3s2p110": ([3, 3, 3], [2, 2, 2], [1, 1, 0], False),
    "conv_k113s112": ([1, 1, 3], [1, 1, 2], [0, 0, 0], False),
}


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden",
                                                                "spconv_*.npz"))))
def test_golden_fixture(cuda, path):
    """fixtures produced by the reference CPU extension (first-encounter output order)."""
    from bevfusion_b200.spconv import ops
    g = np.load(path)
    subm = bool(g["subm"])
    idx = torch.from_numpy(g["indices"]).to(cuda)
    outids, pairs, num = ops.get_indice_pairs(idx, int(g["batch_size"]), list(g["spatial_shape"]),
                                              list(g["ksize"]), list(g["stride"]), list(g["padding"]),
                                              1, 0, subm)
    outids, pairs, num = outids.cpu().numpy(), pairs.cpu().numpy(), num.cpu().numpy()
    out_shape = list(g["out_shape"])
    assert np.array_equal(num, g["indice_num"])                       # bit-exact pair counts
    if subm:
        assert np.array_equal(outids, g["outids"])
        assert pair_sets(pairs, num) == pair_sets(g["indice_pairs"], g["indice_num"])
        order = np.arange(outids.shape[0])
    else:
        # ours: ascending flat index (the reference GPU order); fixture: first-encounter order
        order = np.argsort(oracle.flat_index(g["outids"], out_shape), kind="stable")
        assert np.array_equal(outids, g["outids"][order])             # bit-exact index set + order
        inv = np.empty_like(order); inv[order] = np.arange(order.size)
        ref_sets = [set((i, int(inv[o])) for i, o in s) for s in pair_sets(g["indice_pairs"], g["indice_num"])]
        assert pair_sets(pairs, num) == ref_sets
    out = ops.indice_conv(torch.from_numpy(g["features"]).to(cuda), torch.from_numpy(g["weight"]).to(cuda),
                          torch.from_numpy(pairs).to(cuda), torch.from_numpy(num).to(cuda),
                          outids.shape[0], False, subm).cpu().numpy()
    assert rel_err(out, g["out"][order]) <= 1e-4


@pytest.mark.parametrize("geom", list(GEOMS))
@pytest.mark.parametrize("cin,cout", [(5, 16), (16, 16), (16, 32), (32, 64), (64, 64), (64, 128), (128, 128)])
def test_conv_vs_oracle(cuda, geom, cin, cout):
    from bevfusion_b200.spconv import ops
    ks, st, pd, subm = GEOMS[geom]
    shape, B, n = [40, 36, 11], 2, 6000
    idx = random_sparse(n, shape, B, seed=cin * 1000 + cout)
    rng = np.random.default_rng(7)
    feat = rng.standard_normal((n, cin)).astype(np.float32)
    W = (rng.standard_normal((*ks, cin, cout)) / np.sqrt(cin * 9)).astype(np.float32)
    gold, gids, gshape = oracle.sparse_conv(feat, idx, B, shape, W, ks, st, pd, [1, 1, 1], subm, acc64=True)
    rb, out_shape = ops.get_rulebook(torch.from_numpy(idx).to(cuda), B, shape, ks, st, pd, 1, 0, subm)
    assert out_shape == gshape and rb.n_out == gids.shape[0]
    assert np.array_equal(rb.outids.cpu().numpy(), gids)              # bit-exact outputs + order
    modes = [0] + ([1, 3] if tc_available(cuda) else [])
    for prec in modes:
        out = ops.sparse_conv(torch.from_numpy(feat).to(cuda), torch.from_numpy(W).to(cuda), rb.nbr,
                              rb.n_out, precision=prec).cpu().numpy()
        assert rel_err(out, gold) <= 1e-4, "precision mode %d" % prec


def test_fused_epilogue(cuda):
    from bevfusion_b200.spconv import ops
    ks, st, pd, subm = GEOMS["subm_k3"]
    shape, B, n, cin, cout = [30, 30, 9], 1, 4000, 32, 32
    idx = random_sparse(n, shape, B, seed=1)
    rng = np.random.default_rng(2)
    feat = rng.standard_normal((n, cin)).astype(np.float32)
    W = (rng.standard_normal((*ks, cin, cout)) / 17).astype(np.float32)
    scale = rng.uniform(0.5, 1.5, cout).astype(np.float32)
    shift = rng.standard_normal(cout).astype(np.float32)
    res = rng.standard_normal((n, cout)).astype(np.float32)
    gold, _, _ = oracle.sparse_conv(feat, idx, B, shape, W, ks, st, pd, [1, 1, 1], subm, acc64=True)
    gold = np.maximum(gold.astype(np.float64) * scale + shift + res, 0).astype(np.float32)
    rb, _ = ops.get_rulebook(torch.from_numpy(idx).to(cuda), B, shape, ks, st, pd, 1, 0, subm)
    t = lambda a: torch.from_numpy(a).to(cuda)
    for prec in [0] + ([1] if tc_available(cuda) else []):
        out = ops.sparse_conv(t(feat), t(W), rb.nbr, rb.n_out, t(scale), t(shift), t(res), True, prec)
        assert rel_err(out.cpu().numpy(), gold) <= 1e-4


def test_rulebook_edge_cases(cuda):
    from bevfusion_b200.spconv import ops
    # empty tensor
    rb, shp = ops.get_rulebook(torch.zeros(0, 4, dtype=torch.int32, device=cuda), 1, [8, 8, 4], 3, 2, 1, 1, 0, False)
    assert rb.n_out == 0 and shp == [4, 4, 2]
    # a single voxel in the corner: SubM has only the centre pair; strided conv one output
    one = torch.tensor([[0, 0, 0, 0]], dtype=torch.int32, device=cuda)
    rb, _ = ops.get_rulebook(one, 1, [8, 8, 4], 3, 1, 1, 1, 0, True)
    nbr = rb.nbr.cpu().numpy()
    assert nbr[13, 0] == 0 and (np.delete(nbr[:, 0], 13) == -1).all()
    pairs, num = rb.pairs()
    assert num.cpu().tolist() == [0] * 13 + [1] + [0] * 13
    rb, _ = ops.get_rulebook(one, 1, [8, 8, 4], 3, 2, 1, 1, 0, False)
    assert rb.n_out == 1 and rb.outids.cpu().tolist() == [[0, 0, 0, 0]]
    # fully dense block: every interior voxel has 27 neighbours
    dense = random_sparse(6 * 6 * 6, [6, 6, 6], 1, seed=0)
    rb, _ = ops.get_rulebook(torch.from_numpy(dense).to(cuda), 1, [6, 6, 6], 3, 1, 1, 1, 0, True)
    cnt = (rb.nbr.cpu().numpy() >= 0).sum(0)
    interior = ((dense[:, 1:] > 0) & (dense[:, 1:] < 5)).all(1)
    assert (cnt[interior] == 27).all() and cnt.min() == 8


def test_dense_layouts(cuda):
    from bevfusion_b200.spconv import SparseConvTensor, ops
    shape, B, n, c = [10, 9, 4], 2, 300, 16
    idx = random_sparse(n, shape, B, seed=3)
    feat = np.random.default_rng(1).standard_normal((n, c)).astype(np.float32)
    gold = oracle.dense(feat, idx, B, shape)                               # [B, C, X, Y, Z]
    t = SparseConvTensor(torch.from_numpy(feat).to(cuda), torch.from_numpy(idx).to(cuda), shape, B)
    assert np.array_equal(t.dense().cpu().numpy(), gold)
    zm = ops.sparse_to_dense(t.features, t.indices, B, shape, z_major=True).cpu().numpy()
    # SparseEncoder layout: permute(0,1,4,2,3).view(N, C*D, H, W)  (sparse_encoder.py:126-130)
    assert np.array_equal(zm, gold.transpose(0, 1, 4, 2, 3).reshape(B, c * shape[2], shape[0], shape[1]))


def reference_case_conv(cuda):
    """inputs of test_vs_reference_cuda_extension: indices, features and one filter per geometry"""
    shape, B, n, cin, cout = [64, 60, 13], 2, 20000, 16, 32
    idx = torch.from_numpy(random_sparse(n, shape, B, seed=9)).to(cuda)
    rng = np.random.default_rng(3)
    feat = torch.from_numpy(rng.standard_normal((n, cin)).astype(np.float32)).to(cuda)
    filters = {name: torch.from_numpy((rng.standard_normal((*GEOMS[name][0], cin, cout)) / 12).astype(np.float32)).to(cuda)
               for name in GEOMS}
    return idx, feat, filters, shape, B


def test_vs_reference_cuda_extension(cuda):
    """rulebook + conv of the reference's own GPU path (sparse_conv_ext built for sm_100)."""
    from bevfusion_b200.spconv import ops
    gold = Gold("spconv_conv")
    idx, feat, filters, shape, B = reference_case_conv(cuda)
    for name, (ks, st, pd, subm) in GEOMS.items():
        outids, pairs, num = ops.get_indice_pairs(idx, B, shape, ks, st, pd, 1, 0, subm)
        gold.exact(name + ".outids", outids)                          # same outputs, same order
        gold.exact(name + ".num", num)
        gold.exact(name + ".pairs", pair_table(pairs, num))
        ours = ops.indice_conv(feat, filters[name], pairs, num, outids.shape[0], False, subm)   # drop-in call
        gold.close(name + ".out", ours, 1e-4)


def make_encoder(cuda, sparse_shape, seed=0):
    from bevfusion_b200.sparse_encoder import SparseEncoder
    torch.manual_seed(seed)
    m = SparseEncoder(in_channels=5, sparse_shape=sparse_shape, output_channels=128,
                      encoder_channels=((16, 16, 32), (32, 32, 64), (64, 64, 128), (128, 128)),
                      encoder_paddings=((0, 0, 1), (0, 0, 1), (0, 0, (1, 1, 0)), (0, 0)),
                      block_type="basicblock").to(cuda).eval()
    for mod in m.modules():                                       # non-trivial BN statistics
        if isinstance(mod, torch.nn.BatchNorm1d):
            mod.running_mean.normal_(0, 0.1); mod.running_var.uniform_(0.5, 1.5)
            mod.weight.data.uniform_(0.8, 1.2); mod.bias.data.normal_(0, 0.1)
    return m


def reference_case_encoder(cuda):
    """inputs of test_encoder_fused_vs_modular_vs_reference: encoder, features, batch-sorted coordinates"""
    shape, B = [160, 160, 41], 2
    m = make_encoder(cuda, shape)
    rng = np.random.default_rng(0)
    idx = random_sparse(12000, [160, 160, 40], B, seed=5)
    order = np.lexsort((idx[:, 3], idx[:, 2], idx[:, 1], idx[:, 0]))   # batch-sorted like the caller
    coors = torch.from_numpy(idx[order]).to(cuda)
    feats = torch.from_numpy(rng.standard_normal((coors.shape[0], 5)).astype(np.float32)).to(cuda)
    return m, feats, coors, B


def test_encoder_fused_vs_modular_vs_reference(cuda):
    """whole SparseEncoder on a small grid: fused-epilogue path == module-by-module path, and
    both match the encoder executed with the reference CUDA extension."""
    m, feats, coors, B = reference_case_encoder(cuda)
    with torch.no_grad():
        modular = m(feats, coors, B, fused=False, precision=0)
        fused = m(feats, coors, B, fused=True, precision=0)
    assert tuple(fused.shape) == (B, 256, 20, 20)
    scale = float(modular.abs().max())
    assert float((fused - modular).abs().max()) <= 1e-4 * scale
    Gold("spconv_encoder").close("out", fused, 1e-4)
    if tc_available(cuda):
        with torch.no_grad():
            for prec in (1, 3):                                      # 3xTF32 and BF16x3 (default)
                tc = m(feats, coors, B, fused=True, precision=prec)
                assert float((tc - modular).abs().max()) <= 1e-4 * scale


def test_weight_gradient_is_reproducible(cuda):
    """the filter gradient is summed in a fixed order (per-chunk partials + ordered reduction, no atomics):
    two runs are bit-identical, also when the row count spans many chunks."""
    from bevfusion_b200.spconv import ops
    shape, B, n, cin, cout = [60, 56, 21], 1, 30000, 32, 64
    idx = torch.from_numpy(random_sparse(n, shape, B, seed=21)).to(cuda)
    rb, _ = ops.get_rulebook(idx, B, shape, 3, 1, 1, 1, 0, True)
    g = torch.Generator(device=cuda).manual_seed(0)
    feat = torch.randn(n, cin, device=cuda, generator=g)
    W = torch.randn(27, cin, cout, device=cuda, generator=g) / 30
    gout = torch.randn(n, cout, device=cuda, generator=g)
    for prec in [0] + ([3] if tc_available(cuda) else []):       # SIMT kernel / tensor-core kernel (spconv_wgrad_tc.cu)
        runs = [ops.sparse_conv_backward(feat, W, gout, rb.nbr, precision=prec) for _ in range(3)]
        for din, dw in runs[1:]:
            assert bool(torch.equal(dw, runs[0][1])) and bool(torch.equal(din, runs[0][0]))
        # and it is the right gradient: dW[k] = sum_o f[nbr[k, o]]^T g[o]   (every offset, many row chunks)
        for k in range(27):
            valid = rb.nbr[k] >= 0
            want = feat[rb.nbr[k][valid].long()].double().t() @ gout[valid].double()
            assert float((runs[0][1][k].double() - want).abs().max()) <= 1e-4 * float(want.abs().max()), (prec, k)


def test_native_plan_vs_python_loop(cuda):
    """bevb200_encoder_forward (one native, sync-free call) == the per-conv python loop of the fused path ==
    the exact-fp32 modular path, on a small grid with two samples and unsorted rows."""
    shape, B = [160, 160, 41], 2
    m = make_encoder(cuda, shape)
    assert m.plan() is not None
    rng = np.random.default_rng(3)
    idx = random_sparse(12000, [160, 160, 40], B, seed=9)            # NOT sorted: level 0 keeps the caller's order
    coors = torch.from_numpy(idx).to(cuda)
    feats = torch.from_numpy(rng.standard_normal((coors.shape[0], 5)).astype(np.float32)).to(cuda)
    with torch.no_grad():
        exact = m(feats, coors, B, fused=False, precision=0)
        native = m(feats, coors, B)                                   # default: native plan, bf16x3
        m.native_plan = False
        loop = m(feats, coors, B, fused=True, precision=3)
        m.native_plan = True
    scale = float(exact.abs().max())
    assert float((native - exact).abs().max()) <= 1e-4 * scale
    assert float((native - loop).abs().max()) <= 2e-5 * scale
    assert bool(((native != 0) == (exact != 0)).all())
    st = m.plan().status.cpu().numpy()
    assert st[0] == 0 and st[1] == coors.shape[0] and all(st[1:] > 0)
    # written in place into a channel slice of a wider buffer (fusers/conv.py:16)
    buf = torch.full((B, 80 + 256, 20, 20), 7.0, device=cuda)
    with torch.no_grad():
        m(feats, coors, B, out=buf[:, 80:])
    assert bool((buf[:, :80] == 7.0).all()) and bool(torch.equal(buf[:, 80:], native))


def test_native_plan_device_side_count_and_caps(cuda):
    """rows beyond the device-side voxel count are ignored (no host round trip for the count); tight level
    caps that hold give the same result, caps that truncate raise the overflow flag."""
    shape, B = [96, 96, 41], 1
    m = make_encoder(cuda, shape, seed=4)
    rng = np.random.default_rng(5)
    n = 5000
    idx = random_sparse(n, [96, 96, 40], B, seed=2)
    coors = torch.from_numpy(idx).to(cuda)
    feats = torch.from_numpy(rng.standard_normal((n, 5)).astype(np.float32)).to(cuda)
    with torch.no_grad():
        want = m(feats, coors, B)
        # cap-sized buffers whose tail holds garbage (in-range coordinates that must NOT become voxels)
        junk = torch.from_numpy(random_sparse(3000, [96, 96, 40], B, seed=77)).to(cuda)
        feats_cap = torch.cat([feats, torch.full((3000, 5), 1e3, device=cuda)])
        coors_cap = torch.cat([coors, junk])
        count = torch.tensor([n], dtype=torch.int32, device=cuda)
        got = m(feats_cap, coors_cap, B, num_voxels=count)
    assert bool(torch.equal(got, want))
    plan = m.plan()
    levels = plan.status.cpu().numpy()[1:]
    with torch.no_grad():
        tight = plan.forward(feats, coors, B, level_caps=[0] + [int(v) + 7 for v in levels[1:]])
    assert bool(torch.equal(tight, want)) and not plan.overflowed()
    with torch.no_grad():
        plan.forward(feats, coors, B, level_caps=[0, int(levels[1]) // 2, 0, 0, 0])
    assert plan.overflowed()
    with torch.no_grad():                                              # and the plan recovers
        assert bool(torch.equal(plan.forward(feats, coors, B), want)) and not plan.overflowed()


def test_native_plan_edge_cases(cuda):
    """zero valid rows (device-side count 0), a batch with an empty sample in the middle, and rows whose
    coordinates lie outside the grid (ignored like the per-conv path ignores them)."""
    shape, B = [96, 96, 41], 3
    m = make_encoder(cuda, shape, seed=8)
    rng = np.random.default_rng(9)
    idx = random_sparse(4000, [96, 96, 40], B, seed=12)
    idx = idx[idx[:, 0] != 1]                                           # sample 1 is empty
    # far outside the grid / batch (rows one step outside would still reach border outputs of a strided conv in the
    # reference's scatter formulation -- neither implementation validates coordinates)
    bad = np.array([[0, -7, 5, 5], [2, 300, 0, 0], [0, 3, 3, 90], [3, 1, 1, 1]], np.int32)
    coors = torch.from_numpy(np.concatenate([idx, bad])).to(cuda)
    feats = torch.from_numpy(rng.standard_normal((coors.shape[0], 5)).astype(np.float32)).to(cuda)
    with torch.no_grad():
        native = m(feats, coors, B)
        m.native_plan = False
        loop = m(feats, coors, B, fused=True, precision=3)
        m.native_plan = True
    assert float((native - loop).abs().max()) <= 2e-5 * float(loop.abs().max())
    assert not bool(native[1].any())                                    # the empty sample stays empty
    with torch.no_grad():
        zero = torch.zeros(1, dtype=torch.int32, device=cuda)
        none = m(feats, coors, B, num_voxels=zero)
    assert not bool(none.any())
    assert m.plan().status.cpu().numpy()[1:].tolist() == [0] * 5
    with torch.no_grad():                                               # and n = 0 rows at all
        e = m(feats[:0], coors[:0], B)
    assert tuple(e.shape) == (B, 256, 12, 12) and not bool(e.any())


def test_native_plan_cuda_graph(cuda):
    """the encoder forward has no host synchronisation: it can be captured once and replayed on new
    voxel features / coordinates / counts written into the same buffers."""
    shape, B = [96, 96, 41], 1
    m = make_encoder(cuda, shape, seed=6)
    plan = m.plan()
    cap = 6000
    feats = torch.zeros((cap, 5), device=cuda)
    coors = torch.zeros((cap, 4), dtype=torch.int32, device=cuda)
    count = torch.zeros(1, dtype=torch.int32, device=cuda)
    out = torch.empty((B, 256, 12, 12), device=cuda)      # z: 41 -> 21 -> 11 -> 5 -> 2 ; x, y: 96 -> 12

    def load(seed, n):
        rng = np.random.default_rng(seed)
        idx = random_sparse(n, [96, 96, 40], B, seed=seed)
        f = rng.standard_normal((n, 5)).astype(np.float32)
        coors[:n].copy_(torch.from_numpy(idx).to(cuda)); feats[:n].copy_(torch.from_numpy(f).to(cuda))
        count.fill_(n)
        return torch.from_numpy(f).to(cuda), torch.from_numpy(idx).to(cuda)

    f0, c0 = load(1, 4000)
    with torch.no_grad():
        plan.forward(feats, coors, B, n_voxels_dev=count, out=out)        # warm-up: parameters, workspace, events
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            plan.forward(feats, coors, B, n_voxels_dev=count, out=out)
        for seed, n in ((1, 4000), (2, 5500), (3, 1200)):
            f, c = load(seed, n)
            g.replay()
            torch.cuda.synchronize()
            eager = m(f, c, B)
            assert bool(torch.equal(out, eager)), (seed, n)


def reference_case_lidar(cuda):
    """inputs of test_lidar_branch_full_size: encoder on the C3 grid, voxel means and coordinates"""
    from bevfusion_b200 import synthetic as S
    from bevfusion_b200.voxelize import Voxelization, voxelize_mean
    L = S.LIDAR_C3
    pts = torch.from_numpy(S.lidar_cloud(seed=0)).to(cuda)
    vox = Voxelization(L["voxel_size"], L["point_cloud_range"], L["max_num_points"], L["max_voxels"]).eval()
    feats, coords = voxelize_mean(*vox(pts), 0)
    return make_encoder(cuda, L["sparse_shape"]), feats, coords


def active_cells(out):
    """[B, C, H, W] -> packed bits of the BEV cells with any non-zero channel"""
    return np.packbits((out != 0).any(1).cpu().numpy().reshape(-1))


def test_lidar_branch_full_size(cuda):
    """BASELINE config C3 end to end: voxelize -> mean -> SparseEncoder on the full
    1440x1440x41 grid; layer sizes follow SURVEY.md App. D and the output is finite / sparse."""
    m, feats, coords = reference_case_lidar(cuda)
    assert feats.shape[0] == 160000
    with torch.no_grad():
        out = m(feats, coords, 1)
    assert tuple(out.shape) == (1, 256, 180, 180)
    assert bool(torch.isfinite(out).all())
    nz = (out.abs().sum(1) > 0).float().mean()
    assert 0.05 < float(nz) < 0.9
    # full-size parity: the same encoder run op by op through the reference's own CUDA extension
    gold = Gold("spconv_lidar")
    gold.close("out", out, 1e-4)
    same = np.unpackbits(active_cells(out)) == np.unpackbits(gold["active_cells"])
    assert same.mean() > 0.9999                                                # same active BEV cells


@pytest.mark.parametrize("geom", list(GEOMS))
@pytest.mark.parametrize("cin,cout", [(5, 16), (16, 32), (32, 32), (32, 64), (64, 64), (64, 128), (128, 128)])
def test_backward_vs_oracle(cuda, geom, cin, cout):
    """indice_conv_backward: input and weight gradients vs the float64 oracle (<= 1e-4 rel)."""
    from bevfusion_b200.spconv import ops
    ks, st, pd, subm = GEOMS[geom]
    shape, B, n = [30, 28, 9], 2, 3000
    idx = random_sparse(n, shape, B, seed=cin + 7 * cout)
    rng = np.random.default_rng(11)
    feat = rng.standard_normal((n, cin)).astype(np.float32)
    W = (rng.standard_normal((*ks, cin, cout)) / np.sqrt(cin * 9)).astype(np.float32)
    outids, pairs, num, oshape = oracle.get_indice_pairs(idx, B, shape, ks, st, pd, [1, 1, 1], subm)
    order = np.arange(outids.shape[0]) if subm else np.argsort(oracle.flat_index(outids, oshape), kind="stable")
    g = rng.standard_normal((outids.shape[0], cout)).astype(np.float32)       # grad in ORACLE row order
    gdin, gdw = oracle.indice_conv_backward(feat, W, g, pairs, num)
    rb, _ = ops.get_rulebook(torch.from_numpy(idx).to(cuda), B, shape, ks, st, pd, 1, 0, subm)
    assert np.array_equal(rb.outids.cpu().numpy(), outids[order])
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda)
    for prec in [0] + ([1, 3] if tc_available(cuda) else []):
        din, dw = ops.sparse_conv_backward(t(feat), t(W), t(g[order]), rb.nbr, precision=prec)
        assert rel_err(din.cpu().numpy(), gdin) <= 1e-4, "input grad, precision %d" % prec
        assert rel_err(dw.cpu().numpy(), gdw) <= 1e-4, "weight grad, precision %d" % prec


def reference_case_backward(cuda):
    """inputs of test_backward_vs_reference_cuda_extension: indices, features and one filter per geometry"""
    shape, B, n, cin, cout = [48, 40, 11], 2, 8000, 32, 64
    idx = torch.from_numpy(random_sparse(n, shape, B, seed=4)).to(cuda)
    rng = np.random.default_rng(5)
    feat = torch.from_numpy(rng.standard_normal((n, cin)).astype(np.float32)).to(cuda)
    filters = {name: torch.from_numpy((rng.standard_normal((*GEOMS[name][0], cin, cout)) / 17).astype(np.float32)).to(cuda)
               for name in GEOMS}
    return idx, feat, filters, shape, B


def test_backward_vs_reference_cuda_extension(cuda):
    from bevfusion_b200.spconv import ops
    gold = Gold("spconv_backward")
    idx, feat, filters, shape, B = reference_case_backward(cuda)
    for i, (name, (ks, st, pd, subm)) in enumerate(GEOMS.items()):
        W = filters[name]
        outids, pairs, num = ops.get_indice_pairs(idx, B, shape, ks, st, pd, 1, 0, subm)
        gold.exact(name + ".outids", outids)                          # the rows the gradient is given for
        g = out_grad(outids.shape[0], W.shape[-1], i).to(cuda)
        din, dw = ops.sparse_conv_ext.indice_conv_backward_fp32(feat, W, g, pairs, num, 0, int(subm))
        gold.close(name + ".din", din, 1e-4)
        gold.close(name + ".dw", dw.reshape(W.shape), 1e-4)


def test_module_autograd(cuda):
    """SubMConv3d / SparseConv3d modules in training mode: loss.backward() populates grads that
    match finite sums computed from the oracle backward."""
    from bevfusion_b200 import spconv
    shape, B, n = [20, 18, 7], 1, 900
    idx = random_sparse(n, shape, B, seed=8)
    rng = np.random.default_rng(9)
    feat = torch.from_numpy(rng.standard_normal((n, 16)).astype(np.float32)).to(cuda).requires_grad_(True)
    conv1 = spconv.SubMConv3d(16, 32, 3, padding=1, bias=False).to(cuda).train()
    conv2 = spconv.SparseConv3d(32, 32, 3, stride=2, padding=1, bias=True).to(cuda).train()
    x = spconv.SparseConvTensor(feat, torch.from_numpy(idx).to(cuda), shape, B)
    y = conv2(conv1(x))
    w = torch.randn_like(y.features)
    (y.features * w).sum().backward()
    assert feat.grad is not None and conv1.weight.grad is not None and conv2.weight.grad is not None
    # oracle: chain the two backward passes
    o1, ids1, sh1 = oracle.sparse_conv(feat.detach().cpu().numpy(), idx, B, shape, conv1.weight.detach().cpu().numpy(),
                                       [3] * 3, [1] * 3, [1] * 3, [1] * 3, True)
    oi, p2, n2, os2 = oracle.get_indice_pairs(ids1, B, shape, [3] * 3, [2] * 3, [1] * 3, [1] * 3, False)
    order = np.argsort(oracle.flat_index(oi, os2), kind="stable")
    inv = np.empty_like(order); inv[order] = np.arange(order.size)
    g2 = w.cpu().numpy()[inv]                        # our rows are flat-index ordered; oracle's are first-encounter
    d1, dw2 = oracle.indice_conv_backward(o1, conv2.weight.detach().cpu().numpy(), g2, p2, n2)
    _, p1, n1, _ = oracle.get_indice_pairs(idx, B, shape, [3] * 3, [1] * 3, [1] * 3, [1] * 3, True)
    d0, dw1 = oracle.indice_conv_backward(feat.detach().cpu().numpy(), conv1.weight.detach().cpu().numpy(), d1, p1, n1)
    assert rel_err(conv2.weight.grad.cpu().numpy(), dw2) <= 1e-4
    assert rel_err(conv1.weight.grad.cpu().numpy(), dw1) <= 1e-4
    assert rel_err(feat.grad.cpu().numpy(), d0) <= 1e-4
    assert rel_err(conv2.bias.grad.cpu().numpy(), w.sum(0).cpu().numpy()) <= 1e-5


def test_half_features(cuda):
    """indice_conv_half: fp16 features / filters in, fp16 out, fp32 accumulation inside."""
    from bevfusion_b200.spconv import ops
    ks, st, pd, subm = GEOMS["subm_k3"]
    shape, B, n, cin, cout = [24, 20, 9], 1, 2000, 32, 32
    idx = random_sparse(n, shape, B, seed=12)
    rng = np.random.default_rng(13)
    feat = rng.standard_normal((n, cin)).astype(np.float16)
    W = (rng.standard_normal((*ks, cin, cout)) / 17).astype(np.float16)
    gold, _, _ = oracle.sparse_conv(feat.astype(np.float32), idx, B, shape, W.astype(np.float32), ks, st, pd,
                                    [1, 1, 1], subm)
    outids, pairs, num = ops.get_indice_pairs(torch.from_numpy(idx).to(cuda), B, shape, ks, st, pd, 1, 0, subm)
    out = ops.sparse_conv_ext.indice_conv_half(torch.from_numpy(feat).to(cuda), torch.from_numpy(W).to(cuda),
                                               pairs, num, outids.shape[0], 0, int(subm))
    assert out.dtype == torch.half
    assert rel_err(out.float().cpu().numpy(), gold) <= 2e-3      # one fp16 rounding of the result


def test_previous_kernel_generation_still_correct(cuda):
    """BEVB200_SPCONV_TC_VARIANT=4 (register gather + shuffle transposes, kept for A/B measurements) is
    read once per process, so it is exercised in a child process: same parity bar as the default."""
    import subprocess
    import sys
    if not tc_available(cuda):
        pytest.skip("no tcgen05 path")
    code = r"""
import numpy as np, torch, oracle
from bevfusion_b200.spconv import ops
rng = np.random.default_rng(3)
shape, B, n = [24, 20, 9], 2, 3000
vol = B * shape[0] * shape[1] * shape[2]
flat = rng.choice(vol, size=n, replace=False)
idx = np.stack([flat // (shape[0] * shape[1] * shape[2]), (flat // (shape[1] * shape[2])) % shape[0],
                (flat // shape[2]) % shape[1], flat % shape[2]], 1).astype(np.int32)
dev = torch.device("cuda:0")
for cin, cout in ((16, 32), (64, 64), (128, 128)):
    feat = rng.standard_normal((n, cin)).astype(np.float32)
    W = (rng.standard_normal((3, 3, 3, cin, cout)) / np.sqrt(cin * 9)).astype(np.float32)
    gold, gids, _ = oracle.sparse_conv(feat, idx, B, shape, W, [3] * 3, [1] * 3, [1] * 3, [1] * 3, True, acc64=True)
    rb, _ = ops.get_rulebook(torch.from_numpy(idx).to(dev), B, shape, 3, 1, 1, 1, 0, True)
    for prec in (1, 3):
        out = ops.sparse_conv(torch.from_numpy(feat).to(dev), torch.from_numpy(W).to(dev), rb.nbr, rb.n_out,
                              precision=prec).cpu().numpy()
        err = np.abs(out - gold).max() / np.abs(gold).max()
        assert err <= 1e-4, (cin, cout, prec, err)
print("variant-4 ok")
"""
    env = dict(os.environ, BEVB200_SPCONV_TC_VARIANT="4",
               PYTHONPATH=os.pathsep.join([os.path.dirname(os.path.dirname(os.path.abspath(__file__)))]
                                          + os.environ.get("PYTHONPATH", "").split(os.pathsep)))
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "variant-4 ok" in r.stdout, r.stdout + r.stderr


def test_gather_variants_are_bit_identical(cuda):
    """The operand gather of the generation-6 kernel has two selectable forms -- LDGSTS (default) and the TMA gather4
    producer warp (BEVB200_V6_TMA=1) -- and generation 5 gathers fp32 rows and splits them on the fly
    (BEVB200_SPCONV_TC_VARIANT=5).  They only differ in HOW the same bf16 hi / lo tile reaches the tensor core: results
    must be bit-identical.  The switches are read once per process, so each form runs in a child process and prints a
    checksum; many tiles, low / high neighbour density, SubM and strided rulebooks."""
    import subprocess
    import sys
    if not tc_available(cuda):
        pytest.skip("no tcgen05 path")
    code = r"""
import hashlib, numpy as np, torch
from bevfusion_b200.spconv import ops
dev = torch.device("cuda:0")
h = hashlib.sha256()
for dens, shape in ((0.03, [96, 90, 21]), (0.5, [40, 36, 11])):
    rng = np.random.default_rng(5)
    vol = shape[0] * shape[1] * shape[2]
    flat = np.sort(rng.choice(vol, size=int(vol * dens), replace=False))
    idx = np.stack([np.zeros_like(flat), flat // (shape[1] * shape[2]), (flat // shape[2]) % shape[1], flat % shape[2]],
                   1).astype(np.int32)
    for subm, st in ((True, 1), (False, 2)):
        rb, _ = ops.get_rulebook(torch.from_numpy(idx).to(dev), 1, shape, 3, st, 1, 1, 0, subm)
        for cin, cout in ((16, 16), (16, 32), (32, 32), (64, 64), (64, 128), (128, 128)):
            g = torch.Generator(device=dev).manual_seed(cin + cout)
            f = torch.randn(idx.shape[0], cin, device=dev, generator=g)
            w = torch.randn(27, cin, cout, device=dev, generator=g) / (3 * cin)
            for rep in range(2):
                out = ops.sparse_conv(f, w, rb.nbr, rb.n_out, precision=3)
                h.update(out.cpu().numpy().tobytes())
print("checksum", h.hexdigest())
"""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sums = {}
    for name, extra in (("default", {}), ("tma gather4", {"BEVB200_V6_TMA": "1"}), ("generation 5", {"BEVB200_SPCONV_TC_VARIANT": "5"})):
        env = dict(os.environ, PYTHONPATH=os.pathsep.join([root] + os.environ.get("PYTHONPATH", "").split(os.pathsep)), **extra)
        r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0 and "checksum" in r.stdout, name + ": " + r.stdout + r.stderr
        sums[name] = r.stdout.split("checksum")[1].split()[0]
    assert len(set(sums.values())) == 1, sums


def test_fused_indice_conv_and_half_backward_shims(cuda):
    """the remaining sparse_conv_ext entry points a 3-D model can reach: fused_indice_conv_* (bias in the
    epilogue; fused_spconv_ops.h:28-131) and indice_conv_backward_half (spconv_ops.h:363-456 on halves)."""
    from bevfusion_b200.spconv import ops
    rng = np.random.default_rng(11)
    idx = random_sparse(800, [12, 10, 6], 2, seed=2)
    feat = torch.from_numpy(rng.standard_normal((idx.shape[0], 16)).astype(np.float32)).to(cuda)
    W = torch.from_numpy((rng.standard_normal((3, 3, 3, 16, 32)) / 12).astype(np.float32)).to(cuda)
    bias = torch.from_numpy(rng.standard_normal(32).astype(np.float32)).to(cuda)
    outids, pairs, num = ops.get_indice_pairs(torch.from_numpy(idx).to(cuda), 2, [12, 10, 6], 3, 1, 1, 1, 0, True)
    ext = ops.sparse_conv_ext
    plain = ext.indice_conv_fp32(feat, W, pairs, num, outids.shape[0], 0, 1)
    fused = ext.fused_indice_conv_fp32(feat, W, bias, pairs, num, outids.shape[0], 0, 1)
    assert float((fused - (plain + bias)).abs().max()) <= 1e-6 * float(plain.abs().max())
    fused_h = ext.fused_indice_conv_half(feat.half(), W.half(), bias.half(), pairs, num, outids.shape[0], 0, 1)
    assert fused_h.dtype == torch.half
    assert float((fused_h.float() - fused).abs().max()) <= 2e-2 * float(fused.abs().max())
    g = torch.randn_like(plain)
    din, dw = ext.indice_conv_backward_fp32(feat, W, g, pairs, num, 0, 1)
    din_h, dw_h = ext.indice_conv_backward_half(feat.half(), W.half(), g.half(), pairs, num, 0, 1)
    assert din_h.dtype == torch.half and dw_h.dtype == torch.half and dw_h.shape == W.shape
    assert float((din_h.float() - din).abs().max()) <= 2e-2 * float(din.abs().max())
    assert float((dw_h.float() - dw).abs().max()) <= 2e-2 * float(dw.abs().max())
    with pytest.raises(AttributeError):                         # out-of-scope names: a plain missing attribute
        ext.indice_maxpool_fp32
    assert not hasattr(ext, "get_indice_pairs_2d")
