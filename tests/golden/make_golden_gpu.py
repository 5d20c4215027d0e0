"""Records tests/golden/refgpu_*.npz: what the reference's own CUDA kernels return on the inputs of the
GPU parity tests (see tests/refgold.py for what is stored).

The reference extensions are its bev_pool, voxel_layer and sparse_conv_ext sources compiled unmodified for
sm_100 into oracle/_ref by oracle/build_ref.py (which needs the reference source tree).  Each case takes its
inputs from the `reference_case_*` function of the test that checks it, so the record and the test cannot
drift apart.

Run on a B200, from the repository root, after build():  python tests/golden/make_golden_gpu.py
"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
ROOT = os.path.dirname(TESTS)
sys.path[:0] = [ROOT, TESTS]
import test_bev_pool_gpu as TB  # noqa: E402
import test_spconv_gpu as TS  # noqa: E402
import test_voxelize_gpu as TV  # noqa: E402
from oracle import conv_output_size  # noqa: E402
from oracle.build_ref import load_ref  # noqa: E402
from oracle.reference_pipeline import reference_encoder_forward  # noqa: E402
from refgold import Record  # noqa: E402


def sync(fn, *args):
    """the reference kernels launch on the legacy default stream"""
    torch.cuda.synchronize()
    out = fn(*args)
    torch.cuda.synchronize()
    return out


def gen_bev_pool(cuda):
    ref = load_ref("bev_pool_ext_ref")
    rec = Record()
    args, dims, og = TB.reference_case_kernel(cuda)
    rec.close("forward", sync(ref.bev_pool_forward, *args, *dims))
    rec.exact("backward", sync(ref.bev_pool_backward, og, args[1], args[2], args[3], *dims))
    rec.save("bev_pool_kernel")

    rec = Record()
    plan, x = TB.reference_case_c2(cuda)
    t = plan.tables
    xs = x.reshape(-1, 80)[t.perm[:t.n_kept].long()].contiguous()    # what bev_pool.py:94 hands the kernel
    out = sync(ref.bev_pool_forward, xs, t.geom.contiguous(), t.lengths.contiguous(), t.starts.contiguous(),
               1, 1, 360, 360)
    rec.close("forward", out)
    rec.exact("nonzero", out != 0)
    rec.save("bev_pool_c2")


def gen_voxelize(cuda):
    ref = load_ref("voxel_layer_ref")
    rec = Record()
    pts, vs, cr, mp, mv = TV.reference_case_voxelize()
    p = torch.from_numpy(pts).to(cuda)
    voxels = torch.zeros(mv, mp, pts.shape[1], device=cuda)
    coors = torch.zeros(mv, 3, dtype=torch.int32, device=cuda)
    num = torch.zeros(mv, dtype=torch.int32, device=cuda)
    m = sync(ref.hard_voxelize, p, voxels, coors, num, vs, cr, mp, mv, 3, True)
    rec.value("voxel_num", m)
    rec.exact("coors", coors[:m])
    rec.exact("num_points", num[:m])
    rec.exact("voxels", voxels[:m])
    rec.save("hard_voxelize")

    for reduce_type in ("mean", "max", "sum"):
        rec = Record()
        pts, coors = TV.reference_case_scatter(cuda)
        red, oc, cmap, cnt = sync(ref.dynamic_point_to_voxel_forward, pts, coors, reduce_type)
        rec.exact("out_coors", oc)
        rec.exact("coors_map", cmap)
        rec.exact("count", cnt)
        (rec.exact if reduce_type == "max" else rec.close)("reduced", red)
        grad = torch.zeros_like(pts)
        sync(ref.dynamic_point_to_voxel_backward, grad, TV.scatter_grad(red), pts, red, cmap, cnt, reduce_type)
        (rec.exact if reduce_type == "max" else rec.close)("grad", grad)
        rec.save("dynamic_scatter_" + reduce_type)


def gen_spconv(cuda):
    ref = load_ref("sparse_conv_ext_ref")
    torch.backends.cuda.matmul.allow_tf32 = False       # the reference GEMM is torch::mm_out

    def rulebook(idx, B, shape, ks, st, pd, subm):
        out_shape = shape if subm else conv_output_size(shape, ks, st, pd, [1, 1, 1])
        return sync(ref.get_indice_pairs_3d, idx, B, out_shape, shape, ks, st, pd, [1, 1, 1], [0, 0, 0], int(subm), 0)

    rec = Record()
    idx, feat, filters, shape, B = TS.reference_case_conv(cuda)
    for name, (ks, st, pd, subm) in TS.GEOMS.items():
        outids, pairs, num = rulebook(idx, B, shape, ks, st, pd, subm)
        rec.exact(name + ".outids", outids)
        rec.exact(name + ".num", num)
        rec.exact(name + ".pairs", TS.pair_table(pairs, num))
        rec.close(name + ".out", sync(ref.indice_conv_fp32, feat, filters[name], pairs, num, outids.shape[0], 0, int(subm)))
    rec.save("spconv_conv")

    rec = Record()
    idx, feat, filters, shape, B = TS.reference_case_backward(cuda)
    for i, (name, (ks, st, pd, subm)) in enumerate(TS.GEOMS.items()):
        W = filters[name]
        outids, pairs, num = rulebook(idx, B, shape, ks, st, pd, subm)
        rec.exact(name + ".outids", outids)
        g = TS.out_grad(outids.shape[0], W.shape[-1], i).to(cuda)
        din, dw = sync(ref.indice_conv_backward_fp32, feat, W, g, pairs, num, 0, int(subm))
        rec.close(name + ".din", din)
        rec.close(name + ".dw", dw.reshape(W.shape))
    rec.save("spconv_backward")

    with torch.no_grad():
        rec = Record()
        m, feats, coors, B = TS.reference_case_encoder(cuda)
        rec.close("out", sync(reference_encoder_forward, ref, m, feats, coors, B))
        rec.save("spconv_encoder")

        rec = Record()
        m, feats, coords = TS.reference_case_lidar(cuda)
        out = sync(reference_encoder_forward, ref, m, feats, coords, 1)
        rec.close("out", out)
        rec.value("active_cells", TS.active_cells(out))
        rec.save("spconv_lidar")


if __name__ == "__main__":
    dev = torch.device("cuda:0")
    gen_bev_pool(dev)
    gen_voxelize(dev)
    gen_spconv(dev)
    print(sorted(f for f in os.listdir(HERE) if f.startswith("refgpu_")))
