"""CPU: the C-ABI library loads and exports every symbol the header declares; host-side logic
(shape arithmetic, module structure, argument validation).  No compute calls."""
import numpy as np
import pytest
import torch


def test_library_exports_every_declared_symbol():
    from bevfusion_b200 import _C
    L = _C.lib()
    declared = _C.declared_symbols()
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(L, name), "missing export: " + name
    assert set(declared) == set(_C._SIGNATURES), "ctypes table out of sync with the header"
    assert L.bevb200_version() >= 100


def test_no_cpu_fallback():
    """CPU tensors must raise, not silently compute (north star: no CPU fallback)."""
    from bevfusion_b200.bev_pool import bev_pool, bev_pool_ext
    from bevfusion_b200.voxelize import Voxelization
    from bevfusion_b200.spconv import ops
    with pytest.raises(RuntimeError):
        bev_pool(torch.zeros(4, 16), torch.zeros(4, 4, dtype=torch.long), 1, 1, 2, 2)
    with pytest.raises(RuntimeError):
        bev_pool_ext.bev_pool_forward(torch.zeros(4, 16), torch.zeros(4, 4, dtype=torch.int32),
                                      torch.ones(1, dtype=torch.int32), torch.zeros(1, dtype=torch.int32),
                                      1, 1, 2, 2)
    vox = Voxelization([0.5, 0.5, 0.5], [0, 0, 0, 4, 4, 4], 5, (10, 10)).eval()
    with pytest.raises(RuntimeError):
        vox(torch.zeros(8, 4))
    with pytest.raises(RuntimeError):
        ops.get_indice_pairs(torch.zeros(3, 4, dtype=torch.int32), 1, [4, 4, 4], 3, 1, 1, 1, 0, True)


def test_product_does_not_import_oracle():
    import glob, os, re
    root = os.path.join(os.path.dirname(__file__), "..", "bevfusion_b200")
    for path in glob.glob(os.path.join(root, "**", "*.py"), recursive=True):
        src = open(path).read()
        assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), path


def test_library_reads_only_documented_switches():
    """The native library reads one environment variable, BEVB200_WGRAD_TC (documented in the header), and its
    build defines no preprocessor switches: every kernel path a user can reach is a path the tests cover."""
    import glob, os, re
    from bevfusion_b200 import build
    names = set()
    for path in glob.glob(os.path.join(build.CSRC, "*")):
        names |= set(re.findall(r'"(BEVB200_\w*)"', open(path).read()))
    assert names == {"BEVB200_WGRAD_TC"}
    assert not any(f.startswith("-D") for f in build.FLAGS), build.FLAGS


def test_conv_output_size_matches_reference_formula():
    from bevfusion_b200.spconv import ops
    import oracle
    for shape, k, s, p in [([1440, 1440, 41], [3, 3, 3], [2, 2, 2], [1, 1, 1]),
                           ([360, 360, 11], [3, 3, 3], [2, 2, 2], [1, 1, 0]),
                           ([180, 180, 5], [1, 1, 3], [1, 1, 2], [0, 0, 0])]:
        assert ops.get_conv_output_size(shape, k, s, p, [1, 1, 1]) == oracle.conv_output_size(
            shape, k, s, p, [1, 1, 1])
    assert ops.get_conv_output_size([1440, 1440, 41], [3] * 3, [2] * 3, [1] * 3, [1] * 3) == [720, 720, 21]
    assert ops.get_conv_output_size([180, 180, 5], [1, 1, 3], [1, 1, 2], [0] * 3, [1] * 3) == [180, 180, 2]


def test_sparse_encoder_structure_and_state_dict():
    from bevfusion_b200.sparse_encoder import voxelnet_0p075_encoder
    from bevfusion_b200.spconv import SparseConv3d, SubMConv3d
    from bevfusion_b200.sparse_block import SparseBasicBlock
    m = voxelnet_0p075_encoder()
    sd = m.state_dict()
    # names / shapes of the reference checkpoint layout (sparse_encoder.py:63-97, 214-216)
    assert tuple(sd["conv_input.0.weight"].shape) == (3, 3, 3, 5, 16)
    assert tuple(sd["encoder_layers.encoder_layer1.0.conv1.weight"].shape) == (3, 3, 3, 16, 16)
    assert tuple(sd["encoder_layers.encoder_layer1.2.0.weight"].shape) == (3, 3, 3, 16, 32)
    assert tuple(sd["encoder_layers.encoder_layer3.2.0.weight"].shape) == (3, 3, 3, 64, 128)
    assert tuple(sd["conv_out.0.weight"].shape) == (1, 1, 3, 128, 128)
    assert "encoder_layers.encoder_layer4.1.bn2.running_var" in sd
    convs = [mod for mod in m.modules() if isinstance(mod, (SparseConv3d, SubMConv3d))]
    assert sum(isinstance(c, SubMConv3d) for c in convs) == 17          # 17 SubM + 4 strided
    assert sum(not c.subm for c in convs) == 4
    assert sum(isinstance(b, SparseBasicBlock) for b in m.modules()) == 8
    down3 = m.encoder_layers.encoder_layer3[2][0]
    assert down3.padding == [1, 1, 0] and down3.stride == [2, 2, 2]
    assert m.conv_out[0].kernel_size == [1, 1, 3] and m.conv_out[0].stride == [1, 1, 2]
    bn = m.conv_input[1]
    assert bn.eps == 1e-3 and abs(bn.momentum - 0.01) < 1e-12


def test_gen_dx_bx_matches_reference_arithmetic():
    from bevfusion_b200.bev_pool import gen_dx_bx
    import oracle
    dx, bx, nx = gen_dx_bx([-54.0, 54.0, 0.3], [-54.0, 54.0, 0.3], [-10.0, 10.0, 20.0])
    odx, obx, onx = oracle.gen_dx_bx([-54.0, 54.0, 0.3], [-54.0, 54.0, 0.3], [-10.0, 10.0, 20.0])
    assert np.array_equal(dx.numpy(), odx) and np.array_equal(bx.numpy(), obx)
    assert nx.tolist() == onx.tolist() == [360, 360, 1]


def test_geometry_and_synthetic_shapes():
    from bevfusion_b200 import synthetic as S
    geom, cfg = S.camera_geometry("tiny")
    assert tuple(geom.shape) == (1, 2, 20, 8, 22, 3)
    pts = S.lidar_cloud(seed=0, sweeps=2)
    assert pts.shape[1] == 5 and pts.dtype == np.float32
    assert len(np.arange(*S.CONFIGS["C2"]["dbound"])) == 118


def test_size_queries_of_the_later_entry_points():
    """pure host-side size arithmetic of the C ABI (no device needed)."""
    from bevfusion_b200 import _C
    L = _C.lib()
    # input channels the TF32 tensor-core kernels run with: <= 8 -> 8 (conv_input: 5), else next power of two;
    # BF16X3 (generation 6) takes the rows as they are: its operand-split pass pads to a multiple of 16
    for c_in, want in ((1, 8), (5, 8), (8, 8), (9, 16), (16, 16), (17, 32), (64, 64), (100, 128), (128, 128)):
        for prec in (1, 2):
            assert L.bevb200_spconv_padded_channels(c_in, prec) == want
        assert L.bevb200_spconv_padded_channels(c_in, 3) == c_in
        assert L.bevb200_spconv_padded_channels(c_in, 0) == c_in          # exact-fp32 path: no padding
    assert L.bevb200_spconv_padded_channels(129, 3) == 129                 # no tensor-core form: unchanged
    for c_in, want in ((1, 16), (5, 16), (16, 16), (17, 32), (33, 64), (100, 128), (128, 128), (129, 0)):
        assert L.bevb200_spconv_split_channels(c_in) == want
    # the packed image of a padded shape is the image of the padded channel count
    assert L.bevb200_spconv_packed_weight_bytes(5, 16, 27, 1) == L.bevb200_spconv_packed_weight_bytes(8, 16, 27, 1) > 0
    assert L.bevb200_spconv_packed_weight_bytes(5, 16, 27, 3) == L.bevb200_spconv_packed_weight_bytes(16, 16, 27, 3) > 0
    assert L.bevb200_spconv_split_weight_bytes(5, 16, 27) == L.bevb200_spconv_packed_weight_bytes(5, 16, 27, 3)
    assert L.bevb200_spconv_packed_weight_bytes(64, 48, 27, 3) == 0        # c_out must be 16 / 32 / 64 / 128
    assert L.bevb200_spconv_packed_weight_bytes(64, 64, 28, 3) == 0        # kernel volume <= 27
    assert L.bevb200_spconv_packed_weight_bytes(128, 128, 27, 3) == 27 * 128 * 128 * 2 * 2   # bf16 hi + lo
    assert L.bevb200_spconv_packed_weight_bytes(128, 128, 27, 1) == 27 * 128 * 128 * 2 * 4   # tf32 hi + lo
    assert L.bevb200_depth_rasterize_workspace_bytes(6, 256, 704) == 6 * 256 * 704 * 4
    assert L.bevb200_depth_rasterize_workspace_bytes(0, 256, 704) == 0
    assert L.bevb200_dynamic_scatter_workspace_bytes(300000) > 300000 * (8 + 8 + 4 + 4 + 4 + 4 + 4)
    assert L.bevb200_dynamic_scatter_workspace_bytes(0) > 0
    # sparse-conv backward workspace: transposed weights + (operand images of the tensor-core filter gradient: input rows
    # and out-grad rows at 4 B per element, channels padded to 32 / 64 / 128, + per-chunk partial dW) + the packed W^T
    ws = L.bevb200_spconv_backward_workspace_bytes
    n_in, n_out = 70000, 50000
    for c_in, c_out in ((64, 64), (16, 32), (5, 16), (128, 128)):
        ce_in, ce_out = max(32, c_in if c_in in (64, 128) else 32), max(32, c_out if c_out in (64, 128) else 32)
        images = n_in * ce_in * 4 + n_out * ce_out * 4
        assert ws(n_in, n_out, c_in, c_out, 27) >= 27 * c_in * c_out * 4 + images
        assert ws(2 * n_in, n_out, c_in, c_out, 27) >= ws(n_in, n_out, c_in, c_out, 27) + n_in * ce_in * 4   # grows with n_in
    assert ws(1000, 1000, 48, 48, 27) > 0                                  # no tensor-core form: the SIMT partials
    assert ws(-1, 10, 16, 16, 27) == 0 and ws(10, 10, 0, 16, 27) == 0     # bad sizes


def test_output_view_validation():
    """`out=` targets of the layout kernels: channel slices of a wider buffer are fine, anything that
    is not dense inside a batch item is rejected before a pointer reaches the library."""
    from bevfusion_b200.spconv.ops import _batch_stride_of
    buf = torch.zeros(2, 336, 6, 5)
    assert _batch_stride_of(buf[:, :80], (2, 80, 6, 5)) == 336 * 30
    assert _batch_stride_of(buf[:, 80:], (2, 256, 6, 5)) == 336 * 30
    assert _batch_stride_of(torch.zeros(1, 8, 3, 3), (1, 8, 3, 3)) == 72
    with pytest.raises(ValueError):
        _batch_stride_of(buf[:, :80, :, 1:], (2, 80, 6, 4))                # inner stride broken
    with pytest.raises(ValueError):
        _batch_stride_of(buf[:, :80], (2, 81, 6, 5))                      # wrong shape
    with pytest.raises(ValueError):
        _batch_stride_of(buf[:, :80].double(), (2, 80, 6, 5))             # wrong dtype


def test_no_cpu_fallback_in_the_later_rows():
    from bevfusion_b200.scatter_points import DynamicScatter
    from bevfusion_b200.voxelize import voxel_layer, voxelize_mean_fused
    from bevfusion_b200.vtransform import points_to_depth
    pts, coors = torch.zeros(6, 5), torch.zeros(6, 3, dtype=torch.int32)
    with pytest.raises(RuntimeError):
        DynamicScatter([0.1] * 3, [0, 0, 0, 1, 1, 1], True)(pts, coors)
    with pytest.raises(ValueError):
        voxel_layer.dynamic_point_to_voxel_forward(pts, coors, "median")
    with pytest.raises(RuntimeError):
        voxelize_mean_fused(pts, [0.5] * 3, [0, 0, 0, 4, 4, 4], 5, 10)
    eye = torch.eye(4).view(1, 1, 4, 4)
    with pytest.raises(ValueError):
        points_to_depth([pts], eye, eye, torch.eye(4).view(1, 4, 4), (8, 8), depth_input="histogram")
    with pytest.raises(RuntimeError):
        points_to_depth([pts], eye, eye, torch.eye(4).view(1, 4, 4), (8, 8))
