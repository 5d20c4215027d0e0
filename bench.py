#!/usr/bin/env python
"""bench.py -- frames/sec of the BEVFusion C+L hot path on B200 (one JSON line on stdout).

A "step" is one frame of the hot path named by BASELINE.json's north_star, on synthetic
nuScenes-shaped inputs (bevfusion_b200/synthetic.py, SURVEY.md section 8d):

    bev_pool forward   6 cam x 118 depth x 32 x 88 frustum, C=80 -> 360x360 BEV   (config C2)
    hard_voxelize      ~296 k points x 5, 0.075 m voxels, grid 1440x1440x40        (config C3)
    voxel mean + SparseEncoder (VoxelNet 0.075: 17 SubM + 4 strided sparse convs) -> [256,180,180]

The dense glue networks of the full model (SwinT, FPNs, fuser, SECOND, TransFusion head) are not part
of the hot path: the headline line times the hot path alone (`config.workload` says so) and the `c4`
object of the same line times the whole camera+LiDAR frame with plain-torch glue nets around it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU); every rank runs the same per-frame work on its
own synthetic sample (weak scaling, no data-path collective -- the path shards by sample), the
timed region is bracketed by barrier + cuda synchronize, time = max over ranks.

--dump-outputs DIR writes the two BEV maps the last timed step returned (rank 0) as DIR/camera_bev.npy and
DIR/lidar_bev.npy, float32; the inputs are seeded, so two builds can be compared output for output.

--impl reference times the reference's CPU implementation of the path on the host cores
(oracle/_ref extension for the sparse encoder, the restated QuickCumsum for bev_pool, the C port
for hard_voxelize), each step a bounded sample of the frame (see `sample`).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "frames/sec C+L BEVFusion hot path (bev_pool + hard_voxelize + SparseEncoder)"
WORKLOAD = ("C2+C3 hot path per frame: bev_pool fwd 6-cam 256x704 D=118 C=80 -> 360x360 (N'=1,993,728 rows, "
            "638 MB fp32) + hard_voxelize ~296k pts 0.075 m (1440x1440x40, cap 160k x 10) + voxel mean + "
            "SparseEncoder VoxelNet-0.075 (17 SubM + 4 strided convs) -> [1,256,180,180]; "
            "dense glue nets (SwinT/FPN/fuser/SECOND/TransFusion) not included")


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"],
                    bf16_tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


# ---------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return None
        return dict(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))


def load_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full`
    pass of THIS round's kernels (profiles/r2_traffic.json names the commit it was taken at); None when
    no capture of the benched kernel generation exists -- nothing is measured in this process."""
    p = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f)
    return {}


def bind_to_gpu_numa_node(local_rank):
    """Pin this process to the CPUs of the GPU's NUMA node BEFORE pinned buffers are allocated, so that
    first-touch puts the staging memory on the GPU-local node (8 ranks H2D-copying through one node's
    memory controllers halved the end-to-end rate in round 1).  Returns the node or None."""
    try:
        p = torch.cuda.get_device_properties(local_rank)
        bus = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        with open("/sys/bus/pci/devices/%s/numa_node" % bus) as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
class HotPath:
    """One frame of the hot path through the repo's public API (bevfusion_b200.*).  No call in
    frame() / frame_lift() synchronises with the host: the voxel count and every sparse-conv row count
    stay on the device, so a frame can be captured in a CUDA graph."""

    def __init__(self, device, seed=0, precision=None, cfg_name="C2", lidar=None, lidar_points=None):
        from bevfusion_b200 import synthetic as S
        from bevfusion_b200.bev_pool import BEVPoolPlan
        from bevfusion_b200.sparse_encoder import SparseEncoder, voxelnet_0p075_encoder
        self.S, self.device, self.cfg_name = S, device, cfg_name
        self.geom, cfg = S.camera_geometry(cfg_name, device=device)
        self.cfg = cfg
        self.plan = BEVPoolPlan(self.geom, cfg["xbound"], cfg["ybound"], cfg["zbound"])   # static per calibration
        self.L = dict(lidar or S.LIDAR_C3)
        torch.manual_seed(seed)
        if lidar is None:
            self.encoder = voxelnet_0p075_encoder().to(device).eval()
        else:
            self.encoder = SparseEncoder(in_channels=5, sparse_shape=self.L["sparse_shape"], output_channels=128,
                                         order=("conv", "norm", "act"),
                                         encoder_channels=((16, 16, 32), (32, 32, 64), (64, 64, 128), (128, 128)),
                                         encoder_paddings=((0, 0, 1), (0, 0, 1), (0, 0, (1, 1, 0)), (0, 0)),
                                         block_type="basicblock").to(device).eval()
        self.precision = precision
        pts = S.lidar_cloud(seed=seed) if lidar_points is None else lidar_points
        self.points_host = torch.from_numpy(pts).pin_memory()
        t = self.plan.tables
        self.n_kept, self.n_intervals, self.n_total = t.n_kept, t.n_intervals, t.n_total
        self.feature_shape = (1, cfg["n_cam"], len(np.arange(*cfg["dbound"])), *cfg["feature_size"], cfg["C"])

    def rebuild_plan(self):
        """what a per-sample camera2lidar costs: get_geometry + quantise / filter / rank / sort / intervals again,
        straight from the calibration matrices (the geometry tensor is not materialised)"""
        from bevfusion_b200.bev_pool import BEVPoolPlan
        from bevfusion_b200.vtransform import create_frustum
        cfg = self.cfg
        if getattr(self, "_rig", None) is None:
            self._rig = {k: v.to(self.device) for k, v in self.S.camera_rig(cfg["n_cam"], cfg["image_size"], 1).items()}
            self._frustum = create_frustum(cfg["image_size"], cfg["feature_size"], cfg["dbound"]).to(self.device)
        r = self._rig
        self.plan = BEVPoolPlan.from_cameras(self._frustum, r["camera2lidar_rots"], r["camera2lidar_trans"], r["intrins"],
                                             r["post_rots"], r["post_trans"], cfg["xbound"], cfg["ybound"], cfg["zbound"])

    def rebuild_plan_from_geometry(self):
        from bevfusion_b200.bev_pool import BEVPoolPlan
        self.plan = BEVPoolPlan(self.geom, self.cfg["xbound"], self.cfg["ybound"], self.cfg["zbound"])

    def device_inputs(self, seed=0):
        x = self.S.lifted_features(self.cfg_name, device=self.device, seed=seed)      # 638 MB at C2, > L2
        return x, self.points_host.to(self.device)

    def lift_inputs(self, seed=0, device=None):
        """what the camera branch hands to the view transform in the real model (depth_lss.py:92-97):
        softmax depth [1,N,D,fH,fW] and channels-last context [1,N,fH,fW,C]"""
        g = torch.Generator().manual_seed(seed)
        _, N, D, fH, fW, C = self.feature_shape
        depth = torch.softmax(torch.randn((1, N, D, fH, fW), generator=g), dim=2).contiguous()
        ctx = torch.randn((1, N, fH, fW, C), generator=g)
        if device is None:
            return depth.pin_memory(), ctx.pin_memory()
        return depth.to(device), ctx.to(device)

    def _lidar(self, points, out=None):
        from bevfusion_b200.voxelize import voxelize_mean_fused
        L = self.L
        feats, coords, _, nv = voxelize_mean_fused(points, L["voxel_size"], L["point_cloud_range"],
                                                   L["max_num_points"], L["max_voxels"][1], 0, sync=False)
        with torch.no_grad():
            return self.encoder(feats, coords, 1, precision=self.precision, num_voxels=nv, out=out)

    def frame(self, x, points, timers=None):
        """x [1,6,118,32,88,80] and points [N,5] on the device -> (bev [1,80,360,360], lidar [1,256,180,180]).
        The camera branch (HBM-bound pooling) and the LiDAR branch (voxelize, rulebooks, convs) are independent
        until the fuser: they are issued on two streams, so the pooling kernel overlaps the voxelizer and the first
        rulebook (small kernels that need no shared memory) instead of preceding them."""
        del timers
        cur = torch.cuda.current_stream(self.device)
        side = self._branch_stream()
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            bev = self.plan(x)
        lidar = self._lidar(points)
        cur.wait_stream(side)
        bev.record_stream(cur)
        return bev, lidar

    def _branch_stream(self):
        s = getattr(self, "_side", None)
        if s is None:
            s = self._side = torch.cuda.Stream(device=self.device)
        return s

    def frame_lift(self, depth, ctx, points):
        """the same frame from the camera branch's real outputs: fused lift (x) pool, no 638 MB volume"""
        cur = torch.cuda.current_stream(self.device)
        side = self._branch_stream()
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            bev = self.plan.lift(depth, ctx)
        lidar = self._lidar(points)
        cur.wait_stream(side)
        bev.record_stream(cur)
        return bev, lidar

    def capture(self, fn, *static_inputs):
        """CUDA graph of fn(*static_inputs) (inputs are read from the same buffers at every replay)."""
        s = torch.cuda.Stream(device=self.device)
        s.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(s):
            for _ in range(2):
                fn(*static_inputs)
        torch.cuda.current_stream(self.device).wait_stream(s)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = fn(*static_inputs)
        return g, out

    # algorithmic work per frame (DESIGN.md section "roofline accounting")
    def bev_pool_bytes(self):
        C = self.cfg["C"]
        nx = self.plan.nx
        return 4 * C * self.n_kept + 4 * C * int(nx[0]) * int(nx[1]) * int(nx[2]) + 4 * self.n_kept + 12 * self.n_intervals

    def encoder_work(self, points):
        """per conv: (c_in, c_out, subm, n_out, pairs) from rulebooks built by the modular python ops"""
        from bevfusion_b200 import spconv
        from bevfusion_b200.spconv.conv import SparseConvolution
        from bevfusion_b200.voxelize import voxelize_mean_fused
        L = self.L
        feats, coords, _ = voxelize_mean_fused(points, L["voxel_size"], L["point_cloud_range"], L["max_num_points"],
                                               L["max_voxels"][1], 0)
        convs = []
        hooks = [m.register_forward_pre_hook(lambda mod, inp: convs.append((mod, inp[0])))
                 for m in self.encoder.modules() if isinstance(m, SparseConvolution)]
        prev = self.encoder.native_plan
        self.encoder.native_plan = False
        try:
            with torch.no_grad():
                self.encoder(feats, coords, 1, precision=self.precision)
        finally:
            self.encoder.native_plan = prev
            for h in hooks:
                h.remove()
        rows = []
        for mod, inp in convs:
            rb, _ = mod._rulebook(inp)
            rows.append(dict(c_in=mod.in_channels, c_out=mod.out_channels, subm=bool(mod.subm), n_out=int(rb.n_out),
                             pairs=int((rb.nbr >= 0).sum())))
        del spconv
        return rows, int(feats.shape[0])


DUMP_MAX_ELEMENTS = 7_500_000     # 30 MB of float32 per array: the two BEV maps stay under 64 MB in all


def dump_outputs(directory, arrays):
    """Write each array as <directory>/<name>.npy in float32.  An array of more than DUMP_MAX_ELEMENTS elements
    is written as a fixed sample of its flattened elements (positions drawn from a generator seeded with its
    size), the same positions in every run."""
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float32)
        if a.size > DUMP_MAX_ELEMENTS:
            a = a.reshape(-1)[np.sort(np.random.default_rng(a.size).choice(a.size, DUMP_MAX_ELEMENTS, replace=False))]
        np.save(os.path.join(directory, name + ".npy"), a)


def time_ms(fn, n=20, warm=3):
    for _ in range(warm):
        fn()
    evs = []
    for _ in range(n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        evs.append((a, b))
    torch.cuda.synchronize()
    return statistics.median(a.elapsed_time(b) for a, b in evs)


def graph_time_ms(device, fn, n=20):
    """median CUDA-event time of one replay of fn() captured as a CUDA graph: the kernels of a multi-launch op
    run back to back, without the host's launch gaps between them"""
    s = torch.cuda.Stream(device=device)
    s.wait_stream(torch.cuda.current_stream(device))
    with torch.cuda.stream(s):
        for _ in range(2):
            fn()
    torch.cuda.current_stream(device).wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        keep = fn()
    ms = time_ms(g.replay, n=n)
    del keep, g
    return ms


def conv_kernel_times(hp, points, frames=3, backward=False):
    """CUDA-event time of the encoder's sparse-conv kernel launches, one by one: the native plan runs the
    convs back to back on one stream, so each conv is re-run alone here through the same C entry point
    (bevb200_spconv_forward_split) on the plan's real rulebooks.  Returns (ms per frame over the conv
    launches, launches per frame, per-layer rows)."""
    from bevfusion_b200 import _C
    rows, _ = hp.encoder_work(points)
    lib = _C.lib()
    dev = hp.device
    from bevfusion_b200 import spconv
    from bevfusion_b200.spconv.conv import SparseConvolution
    from bevfusion_b200.voxelize import voxelize_mean_fused
    L = hp.L
    feats, coords, _ = voxelize_mean_fused(points, L["voxel_size"], L["point_cloud_range"], L["max_num_points"],
                                           L["max_voxels"][1], 0)
    convs = []
    hooks = [m.register_forward_pre_hook(lambda mod, inp: convs.append((mod, inp[0])))
             for m in hp.encoder.modules() if isinstance(m, SparseConvolution)]
    hp.encoder.native_plan = False
    try:
        with torch.no_grad():
            hp.encoder(feats, coords, 1, precision=hp.precision)
    finally:
        hp.encoder.native_plan = True
        for h in hooks:
            h.remove()
    total, per_layer = 0.0, []
    bwd_total = [0.0]
    for (mod, inp), row in zip(convs, rows):
        rb, _ = mod._rulebook(inp)
        cin, cout, kv = mod.in_channels, mod.out_channels, rb.nbr.shape[0]
        n_in = inp.features.shape[0]
        ce = lib.bevb200_spconv_split_channels(cin)
        fs = torch.empty((n_in, ce * 4), dtype=torch.uint8, device=dev)
        _C.check(lib.bevb200_spconv_split_rows(_C.ptr(inp.features.contiguous()), n_in, 0, cin, _C.ptr(fs),
                                               _C.current_stream(dev)), "split_rows")
        w = mod.weight.detach().float().contiguous()
        pk = torch.empty(lib.bevb200_spconv_split_weight_bytes(cin, cout, kv), dtype=torch.uint8, device=dev)
        _C.check(lib.bevb200_spconv_pack_split_weights(_C.ptr(w), cin, cout, kv, _C.ptr(pk), _C.current_stream(dev)), "pack")
        out = torch.empty((rb.n_out, cout), dtype=torch.float32, device=dev)
        osp = torch.empty((rb.n_out, cout * 4), dtype=torch.uint8, device=dev)
        scale = torch.ones(cout, device=dev)

        def run():
            _C.check(lib.bevb200_spconv_forward_split(_C.ptr(fs), _C.ptr(pk), _C.ptr(rb.nbr), rb.n_out, n_in, rb.n_out, 0,
                                                      ce, cout, kv, _C.ptr(scale), _C.ptr(scale), 0, 1, _C.ptr(out),
                                                      _C.ptr(osp), _C.current_stream(dev)), "forward_split")
        ms = time_ms(run, n=frames * 3, warm=2)
        total += ms
        entry = dict(row, us=round(ms * 1e3, 1), tflops=round(2.0 * row["pairs"] * cin * cout / (ms * 1e-3) / 1e12, 2))
        if backward:
            # training side (spconv_ops.h:363-456): input gradient = the forward kernel on the transposed table,
            # filter gradient = chunked outer products + ordered reduction (no atomics)
            from bevfusion_b200.spconv import ops as sp_ops
            nbr_t = sp_ops.transpose_nbr(rb.nbr, n_in)
            gout = torch.randn(rb.n_out, cout, device=dev)
            feats_f = inp.features.contiguous()
            bms = time_ms(lambda: sp_ops.sparse_conv_backward(feats_f, w, gout, rb.nbr, nbr_t), n=3, warm=1)
            entry["backward_us"] = round(bms * 1e3, 1)
            bwd_total[0] += bms
            del nbr_t, gout
        per_layer.append(entry)
    del spconv
    if backward:
        return total, len(convs), per_layer, bwd_total[0]
    return total, len(convs), per_layer


def gpu_reference_leg(hp, x, pts):
    """The reference's own CUDA kernels (oracle/_ref: its extensions compiled unmodified for sm_100) timed on
    this GPU on the same inputs: bev_pool_forward on sorted rows (bev_pool_cuda.cu:20-42), deterministic
    hard_voxelize (voxelization_cuda.cu:231-373), SparseEncoder through get_indice_pairs_3d + indice_conv_fp32
    (spconv_ops.h:27-141, 260-361).  Run after the timed region; a reported baseline, like cpu_baseline."""
    try:
        from oracle.build_ref import built, load_ref
        from oracle import reference_pipeline as RP
    except Exception as e:                                    # pragma: no cover
        return {"unavailable": "oracle import failed: %s" % e}
    need = ("bev_pool_ext_ref", "voxel_layer_ref", "sparse_conv_ext_ref")
    if not all(built(n) for n in need):
        return {"unavailable": "oracle/_ref is not built"}
    dev = hp.device
    out = {}
    t = hp.plan.tables
    Bq, Dq, Hq, Wq = t.dims
    C = hp.cfg["C"]
    bev = load_ref("bev_pool_ext_ref")
    xs = x.reshape(-1, C)[t.perm[:t.n_kept].long()].contiguous()

    def wall_ms(fn, n=3):
        fn(); torch.cuda.synchronize()
        ts = []
        for _ in range(n):
            torch.cuda.synchronize(); t0 = time.perf_counter(); fn(); torch.cuda.synchronize()
            ts.append((time.perf_counter() - t0) * 1e3)
        return statistics.median(ts)

    # the reference kernel launches on the legacy default stream (bev_pool_cuda.cu:88): time with host clocks
    out["bev_pool_forward_ms"] = round(wall_ms(lambda: bev.bev_pool_forward(xs, t.geom, t.lengths, t.starts, Bq, Dq, Hq, Wq), 5), 4)
    out["bev_pool_sort_gather_ms"] = round(wall_ms(lambda: x.reshape(-1, C)[t.perm[:t.n_kept].long()], 3), 4)
    del xs
    L = hp.L
    vl = load_ref("voxel_layer_ref")
    mv, mp = L["max_voxels"][1], L["max_num_points"]

    def ref_vox():
        voxels = pts.new_zeros((mv, mp, pts.shape[1]))
        coors = pts.new_zeros((mv, 3), dtype=torch.int)
        num = pts.new_zeros((mv,), dtype=torch.int)
        n = vl.hard_voxelize(pts, voxels, coors, num, L["voxel_size"], L["point_cloud_range"], mp, mv, 3, True)
        return voxels[:n], coors[:n], num[:n]
    out["hard_voxelize_ms"] = round(wall_ms(ref_vox, 3), 3)
    v, c, n = ref_vox()
    feats = v.sum(dim=1) / n.type_as(v).view(-1, 1)
    coords = torch.nn.functional.pad(c, (1, 0), mode="constant", value=0)
    sp = load_ref("sparse_conv_ext_ref")
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True              # the reference era's default (torch 1.9-1.11)
    try:
        with torch.no_grad():
            out["sparse_encoder_ms"] = round(wall_ms(lambda: RP.reference_encoder_forward(sp, hp.encoder, feats, coords, 1), 3), 3)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    out["frame_ms"] = round(out["bev_pool_forward_ms"] + out["bev_pool_sort_gather_ms"] + out["hard_voxelize_ms"]
                            + out["sparse_encoder_ms"], 3)
    out["note"] = ("reference CUDA kernels recompiled for sm_100, host-clock medians incl. their own device syncs; "
                   "bev_pool = forward kernel on pre-sorted rows + the x[kept][argsort] gather the reference does per "
                   "call (bev_pool.py:94; sort time not included); encoder = reference rulebook + gather/cuBLAS(TF32 "
                   "allowed)/scatter per offset with torch BN/ReLU")
    return out


def c4_leg(hp, device, steps, warmup, world):
    """BASELINE config C4: the full camera+LiDAR frame -- plain-torch glue nets (tools/c4_glue.py, cuDNN /
    cuBLAS, TF32 allowed like the reference era's defaults, random frozen weights) around this repo's hot
    path: LiDAR depth images -> dtransform/depthnet -> fused lift (x) bev_pool, hard voxelize + mean ->
    SparseEncoder written in place into the fuser input, fuser -> SECOND -> SECONDFPN -> TransFusion head.
    Camera and LiDAR branches run on two streams.  FPS protocol of tools/benchmark.py:56-85 (per-frame
    wall clock bracketed by synchronize) is replaced by CUDA events over `steps` frames."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import c4_glue
    from bevfusion_b200 import synthetic as S
    from bevfusion_b200.vtransform import points_to_depth
    prev = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        torch.manual_seed(0)
        glue = c4_glue.GlueNets().to(device).eval()
        M = S.lidar_camera_matrices(6, (256, 704), batch=1, augment=False)
        l2i, ia, la = (M[k].to(device) for k in ("lidar2image", "img_aug_matrix", "lidar_aug_matrix"))
        img = torch.randn(1, 6, 3, 256, 704, device=device)
        pts = hp.points_host.to(device)
        fuser_in = torch.zeros(1, 80 + 256, 180, 180, device=device)
        cam_stream, lid_stream = torch.cuda.Stream(device=device), torch.cuda.Stream(device=device)
        marks = {}

        def frame(timed=False):
            def mark(name, stream):
                if timed:
                    e = torch.cuda.Event(enable_timing=True)
                    e.record(stream)
                    marks.setdefault(name, []).append(e)
            main = torch.cuda.current_stream(device)      # the capturing stream when the frame is recorded as a graph
            with torch.no_grad():
                mark("t0", main)
                cam_stream.wait_stream(main); lid_stream.wait_stream(main)
                with torch.cuda.stream(lid_stream):
                    hp._lidar(pts, out=fuser_in[:, 80:])
                    mark("lidar_done", lid_stream)
                with torch.cuda.stream(cam_stream):
                    feat = glue.camera_features(img)                                   # SwinT + FPN
                    mark("camera_nets", cam_stream)
                    d = points_to_depth([pts], l2i, ia, la, (256, 704))              # [1,6,1,256,704]
                    depth, ctx = glue.lss.lift_inputs(feat, d.flatten(0, 1))
                    cam_bev = hp.plan.lift(depth.view(1, 6, *depth.shape[1:]), ctx.view(1, 6, *ctx.shape[1:]))
                    mark("view_transform", cam_stream)
                main.wait_stream(cam_stream); main.wait_stream(lid_stream)
                boxes, scores, labels = glue.decode(cam_bev, fuser_in)
                mark("decode", main)
                return boxes, scores, labels

        for _ in range(max(warmup, 3)):
            frame()
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = frame(True)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms], dtype=torch.float64, device=device)
        if world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms = float(t.item()) / steps

        def span(a, b):
            return round(statistics.mean(x.elapsed_time(y) for x, y in zip(marks[a], marks[b])), 3)
        res = {"frames_per_s": round(world * 1000.0 / ms, 2), "ms_per_frame": round(ms, 3), "steps": steps,
               "n_gpus": world, "boxes": list(out[0].shape),
               "stages_ms": {"lidar_branch(voxelize+SparseEncoder, own stream)": span("t0", "lidar_done"),
                             "camera_nets(SwinT+FPN)": span("t0", "camera_nets"),
                             "depth_images+depthnet+lift_pool": span("camera_nets", "view_transform"),
                             "downsample+fuser+SECOND+FPN+TransFusion": span("view_transform", "decode")},
               "glue": "plain torch fp32 tensors, TF32 allowed for cuDNN / cuBLAS, random frozen weights, eval-mode BN; "
                       "37 M parameters; eager launches (not graph-captured)",
               "target": ">= 25 frames/s on 1 GPU (BASELINE.json north_star)"}
        # the same frame recorded once as a CUDA graph (static image / point buffers) and replayed: what a deployment
        # does, and possible because nothing in the hot path synchronises with the host
        try:
            side = torch.cuda.Stream(device=device)
            side.wait_stream(torch.cuda.current_stream(device))
            with torch.cuda.stream(side):
                frame()
            torch.cuda.current_stream(device).wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                gout = frame()
            for _ in range(3):
                g.replay()
            torch.cuda.synchronize()
            if world > 1:
                torch.distributed.barrier()
            e0.record()
            for _ in range(steps):
                g.replay()
            e1.record()
            torch.cuda.synchronize()
            t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=device)
            if world > 1:
                torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            gms = float(t.item()) / steps
            same = bool(torch.equal(gout[0], out[0]))
            res["graph"] = {"frames_per_s": round(world * 1000.0 / gms, 2), "ms_per_frame": round(gms, 3),
                            "boxes_equal_to_eager": same}
            del g, gout
        except Exception as exc:                       # a glue op that cannot be captured: report, keep the eager line
            res["graph"] = {"unavailable": "%s: %s" % (type(exc).__name__, str(exc)[:200])}
            if world > 1:                              # keep the ranks' collectives aligned
                pass
        del glue
        return res
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev
        torch.cuda.empty_cache()


def c5_leg(device, peaks):
    """BASELINE configs[4], the high-resolution stress case: 6 cam 512x1408 -> 64x176, D=200, C=80 -> 256x256 BEV
    (13.5 M rows, 4.3 GB of lifted features) and a 0.05 m voxel grid (2160x2160x41)."""
    from bevfusion_b200 import synthetic as S
    lidar = dict(voxel_size=[0.05, 0.05, 0.2], point_cloud_range=[-54.0, -54.0, -5.0, 54.0, 54.0, 3.0],
                 max_num_points=10, max_voxels=(120000, 240000), sparse_shape=[2160, 2160, 41])
    hp = HotPath(device, seed=0, cfg_name="C5", lidar=lidar)
    x, pts = hp.device_inputs(seed=0)
    pool_ms = time_ms(lambda: hp.plan.pool(x), n=10)
    call_ms = time_ms(lambda: hp.plan(x), n=10)
    nbytes = hp.bev_pool_bytes()
    depth, ctx = hp.lift_inputs(seed=0, device=device)
    lift_ms = graph_time_ms(device, lambda: hp.plan.lift(depth, ctx), n=10)
    del x, depth, ctx
    lid_ms = time_ms(lambda: hp._lidar(pts), n=10)
    rows, n_vox = hp.encoder_work(pts)
    flops = sum(2 * r["pairs"] * r["c_in"] * r["c_out"] for r in rows)
    gbs = nbytes / (pool_ms * 1e-3) / 1e9
    res = {"workload": "C5: bev_pool 6-cam 512x1408 D=200 C=80 -> 256x256 (N'=%d rows, %.2f GB fp32); hard_voxelize 0.05 m "
                       "(2160x2160x40, cap 240k) + SparseEncoder on [2160,2160,41]" % (hp.n_total, hp.n_total * 320 / 1e9),
           "bev_pool": {"kept_rows": hp.n_kept, "intervals": hp.n_intervals, "pool_ms": round(pool_ms, 4),
                        "pool_plus_layout_ms": round(call_ms, 4), "algorithmic_bytes": nbytes, "GBs": round(gbs, 1),
                        "frac_of_hbm_peak": round(gbs / peaks["hbm_gbs"], 4), "fused_lift_pool_ms": round(lift_ms, 4)},
           "lidar": {"voxels": n_vox, "voxelize_plus_encoder_ms": round(lid_ms, 4), "encoder_gflop": round(flops / 1e9, 1),
                     "rows_per_level": [r["n_out"] for r in rows if not r["subm"]]}}
    del hp
    torch.cuda.empty_cache()
    return res


def run_ours(args, rank, world, local_rank):
    from bevfusion_b200 import _C
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank)
    _C.lib()
    peaks = load_peaks()
    traffic = load_traffic()
    hp = HotPath(device, seed=rank, precision=args.precision)
    x, pts = hp.device_inputs(seed=rank)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        t = torch.tensor([ms], dtype=torch.float64, device=device)
        if world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return float(t.item())

    warm = max(args.warmup, 3)
    for _ in range(warm):
        out = hp.frame(x, pts)
    del out
    barrier()
    # --- device-resident throughput: the frame as ONE CUDA graph (no host sync anywhere in it) -------
    graph, gout = hp.capture(hp.frame, x, pts)
    for _ in range(warm):
        graph.replay()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:          # one nvidia-smi poller per job (its driver queries can stall CUDA calls)
        sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        graph.replay()
    e1.record()
    barrier()
    ms_per_step = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    # what the last timed replay returned, copied out after the timed region
    outputs = {"camera_bev": gout[0].cpu().numpy(), "lidar_bev": gout[1].cpu().numpy()} if args.dump_outputs else None
    # --- stage times: each stage as its own graph, replayed back to back with events between them -------
    from bevfusion_b200.voxelize import voxelize_mean_fused
    L = hp.L

    def vox_only():
        return voxelize_mean_fused(pts, L["voxel_size"], L["point_cloud_range"], L["max_num_points"], L["max_voxels"][1], 0,
                                   sync=False)
    g_bev, o_bev = hp.capture(hp.plan, x)
    g_vox, o_vox = hp.capture(vox_only)

    def enc_only():
        with torch.no_grad():
            return hp.encoder(o_vox[0], o_vox[1], 1, precision=hp.precision, num_voxels=o_vox[3])
    g_enc, o_enc = hp.capture(enc_only)
    marks = []
    n_stage = max(10, min(args.steps, 50))
    for _ in range(n_stage):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record(); g_bev.replay(); ev[1].record(); g_vox.replay(); ev[2].record(); g_enc.replay(); ev[3].record()
        marks.append(ev)
    torch.cuda.synchronize()
    stages = dict(bev_pool_ms=statistics.median(m[0].elapsed_time(m[1]) for m in marks),
                  voxelize_ms=statistics.median(m[1].elapsed_time(m[2]) for m in marks),
                  encoder_ms=statistics.median(m[2].elapsed_time(m[3]) for m in marks))
    del g_bev, g_vox, g_enc, o_bev, o_enc
    # --- the same frames launched eagerly from python (what round 1 timed) -------------------------------
    _C.reset_launch_count()
    barrier()
    e0.record()
    for _ in range(args.steps):
        out = hp.frame(x, pts)
    e1.record()
    barrier()
    launches = _C.launch_count()
    clocks = sampler.stop()
    eager_ms = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    del out, o_vox
    # --- per-sample calibration: the pooling plan rebuilt every frame -----------------------------------
    prepare_geom_ms = time_ms(hp.rebuild_plan_from_geometry, n=5, warm=1)
    prepare_ms = time_ms(hp.rebuild_plan, n=5, warm=1)

    def frame_rebuild():
        hp.rebuild_plan()
        hp.frame(x, pts)
    barrier()
    rebuild_ms = max_over_ranks(time_ms(frame_rebuild, n=max(3, min(args.steps, 10)), warm=1))
    del graph, gout

    # --- end to end through the public API with HOST buffers ------------------------------------------
    # (a) `e2e`: the inputs the view transform really gets -- softmax depth + context from the camera branch
    #     (13.4 MB) and the point cloud (5.9 MB) -- through the fused lift; (b) `e2e_materialised`: the 638 MB
    #     lifted volume of the drop-in bev_pool contract.  H2D of frame i+1 overlaps the compute of frame i.
    copy_stream = torch.cuda.Stream(device=device)
    main_stream = torch.cuda.current_stream(device)
    bev_h = torch.empty((1, 80, 360, 360), dtype=torch.float32).pin_memory()
    lid_h = torch.empty((1, 256, 180, 180), dtype=torch.float32).pin_memory()

    out_stream = torch.cuda.Stream(device=device)

    def e2e_pipeline(host_tensors, compute, nframes):
        """three streams: H2D of frame i+1 (copy stream), compute of frame i (main), D2H of frame i-1 (out stream).
        The compute of each of the two input buffer sets is captured once as a CUDA graph (the API is sync-free, so a
        user can do exactly that) and replayed per frame; every frame still copies its inputs in and its results out."""
        bufs = [[torch.empty(h.shape, dtype=h.dtype, device=device) for h in host_tensors] for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]
        freed = [torch.cuda.Event() for _ in range(2)]
        out_done = [torch.cuda.Event() for _ in range(2)]
        done = torch.cuda.Event()
        for bset in bufs:                                   # defined inputs for the capture's warm-up runs
            for dst, src in zip(bset, host_tensors):
                dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
        graphs = [hp.capture(compute, *bset) for bset in bufs]

        def stage_in(i):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(freed[i % 2])
                for dst, src in zip(bufs[i % 2], host_tensors):
                    dst.copy_(src, non_blocking=True)
                ready[i % 2].record(copy_stream)

        def run(n):
            for f in freed:
                f.record(main_stream)
            for f in out_done:
                f.record(out_stream)
            stage_in(0)
            for i in range(n):
                if i + 1 < n:
                    stage_in(i + 1)
                main_stream.wait_event(ready[i % 2])
                main_stream.wait_event(out_done[i % 2])   # this graph's output buffers have been read out
                g, (bev, lidar) = graphs[i % 2]
                g.replay()
                freed[i % 2].record(main_stream)
                done.record(main_stream)
                with torch.cuda.stream(out_stream):       # D2H of the step's results
                    out_stream.wait_event(done)
                    bev_h.copy_(bev, non_blocking=True)
                    lid_h.copy_(lidar, non_blocking=True)
                    out_done[i % 2].record(out_stream)
            main_stream.wait_stream(out_stream)

        run(2)
        barrier()
        e0.record()
        run(nframes)
        e1.record()
        barrier()
        ms = max_over_ranks(e0.elapsed_time(e1)) / nframes
        del graphs
        return ms

    dh, ch = hp.lift_inputs(seed=rank)
    ph = hp.points_host
    e2e_steps = max(3, min(args.steps, 20))
    e2e_ms = e2e_pipeline([dh, ch, ph], hp.frame_lift, e2e_steps)
    h2d = (dh.numel() + ch.numel() + ph.numel()) * 4
    d2h = (bev_h.numel() + lid_h.numel()) * 4
    del x
    torch.cuda.empty_cache()
    xh = torch.empty(hp.feature_shape, dtype=torch.float32).pin_memory()
    block = torch.randn(hp.feature_shape[2:], generator=torch.Generator().manual_seed(rank))
    for cam in range(hp.feature_shape[1]):
        xh[0, cam].copy_(block + 0.01 * cam)
    mat_steps = max(3, min(args.steps, 6))
    e2e_mat_ms = e2e_pipeline([xh, ph], hp.frame, mat_steps)
    h2d_mat = (xh.numel() + ph.numel()) * 4
    del xh, block
    torch.cuda.empty_cache()

    # --- C4: the full camera+LiDAR frame with the plain-torch glue nets (all ranks, weak scaling) --------
    c4 = None if args.no_c4 else c4_leg(hp, device, max(5, min(args.steps, 20)), 3, world)

    if rank != 0:
        return
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
        del outputs
    # --- roofline of the dominant kernel + the north star's named kernel (bev_pool) --------
    x, pts = hp.device_inputs(seed=0)
    rows, n_vox = hp.encoder_work(pts)
    flops = sum(2 * r["pairs"] * r["c_in"] * r["c_out"] for r in rows)
    pairs = sum(r["pairs"] for r in rows)
    pool_bytes = hp.bev_pool_bytes()
    # bev_pool alone, CUDA events, inputs (638 / 588 MB) larger than L2:
    #   plan path   = interval-cell kernel + pooling kernel reading rows through perm (gather + zero-fill fused) + fix-up
    #   drop-in op  = memset + pooling kernel + fix-up on already sorted rows (the reference contract)
    from bevfusion_b200.bev_pool import bev_pool_ext, _PoolPerm
    t = hp.plan.tables
    pool_eager_ms = time_ms(lambda: hp.plan.pool(x))
    pool_ms = graph_time_ms(device, lambda: hp.plan.pool(x))
    xs = x.reshape(-1, 80)[t.perm[:t.n_kept].long()].contiguous()
    Bq, Dq, Hq, Wq = t.dims
    op_ms = graph_time_ms(device, lambda: bev_pool_ext.bev_pool_forward(xs, t.geom, t.lengths, t.starts, Bq, Dq, Hq, Wq))
    del xs
    og = torch.randn(Bq, Dq, Hq, Wq, 80, device=device)

    class _Ctx:
        tables, c = t, 80
    bwd_ms = time_ms(lambda: _PoolPerm.backward(_Ctx, og))
    bwd_bytes = 4 * 80 * t.n_intervals + 4 * 80 * t.n_total + 4 * t.n_total
    depth, ctx = hp.lift_inputs(seed=0, device=device)
    lift_ms = graph_time_ms(device, lambda: hp.plan.lift_pool(depth, ctx))
    os.environ["BEVB200_LIFT_VARIANT"] = "rows"            # the round-1 kernel: one context-row gather per kept point
    try:
        lift_rows_ms = graph_time_ms(device, lambda: hp.plan.lift_pool(depth, ctx))
    finally:
        del os.environ["BEVB200_LIFT_VARIANT"]
    t0 = time.perf_counter()
    hp.plan._lift_cache = None
    hp.plan.lift_pool(depth, ctx)
    torch.cuda.synchronize()
    lift_prepare_ms = (time.perf_counter() - t0) * 1e3 - lift_ms
    del og, depth, ctx
    # SURVEY.md section 8(f) rows (timed alone, CUDA events, median of 20):
    from bevfusion_b200 import synthetic as S_
    from bevfusion_b200.scatter_points import dynamic_scatter
    from bevfusion_b200.voxelize import voxel_layer, voxelize_mean, voxelize_mean_fused
    from bevfusion_b200.vtransform import points_to_depth
    L_ = S_.LIDAR_C3
    fused_vox_ms = graph_time_ms(device, lambda: voxelize_mean_fused(pts, L_["voxel_size"], L_["point_cloud_range"], 10, 160000, 0, sync=False))
    unfused_vox_ms = time_ms(lambda: voxelize_mean(*hp_voxelize(pts, L_), 0))
    dcoors = torch.zeros(pts.shape[0], 3, dtype=torch.int32, device=device)
    voxel_layer.dynamic_voxelize(pts, dcoors, L_["voxel_size"], L_["point_cloud_range"], 3)
    scatter_ms = time_ms(lambda: dynamic_scatter(pts, dcoors, "mean"))
    M_ = S_.lidar_camera_matrices(6, (256, 704), batch=1)
    margs = (M_["lidar2image"].to(device), M_["img_aug_matrix"].to(device), M_["lidar_aug_matrix"].to(device), (256, 704))
    depth_ms = graph_time_ms(device, lambda: points_to_depth([pts], *margs))
    next_rows = {"voxelize_mean_fused_ms": round(fused_vox_ms, 4), "voxelize_then_mean_ms": round(unfused_vox_ms, 4),
                 "dynamic_scatter_mean_ms": round(scatter_ms, 4), "lidar_depth_images_6x256x704_ms": round(depth_ms, 4),
                 "points": int(pts.shape[0]),
                 "note": "voxelize_mean_fused is the sync-free variant frame() uses (count stays on the device); "
                         "voxelize_then_mean / dynamic_scatter include their host-side result-size readback"}
    pool_gbs = pool_bytes / (pool_ms * 1e-3) / 1e9
    op_gbs = pool_bytes / (op_ms * 1e-3) / 1e9
    enc_tflops = flops / (stages["encoder_ms"] * 1e-3) / 1e12
    roof_pool = dict(kernel="bevpool_fwd_tma_kernel<20,PERM> (plan API: gather through perm + zero-fill fused; + cells, fix-up)",
                     bound="hbm", achieved=round(pool_gbs, 1), peak=peaks["hbm_gbs"], unit="GB/s",
                     frac=round(pool_gbs / peaks["hbm_gbs"], 4), traffic=traffic.get("bev_pool_plan_bytes"),
                     ms=round(pool_ms, 4), ms_eager_launches=round(pool_eager_ms, 4), algorithmic_bytes=pool_bytes,
                     peak_source=peaks["source"],
                     timing="CUDA events around one graph replay of the op's kernels (cells + pooling + fix-up), median of 20; "
                            "x (638 MB) is larger than L2")
    roof_pool_op = dict(kernel="bevpool_fwd_tma_kernel<20,SORTED> (drop-in bev_pool_forward on sorted rows; + memset, fix-up)",
                        bound="hbm", achieved=round(op_gbs, 1), peak=peaks["hbm_gbs"], unit="GB/s",
                        frac=round(op_gbs / peaks["hbm_gbs"], 4), traffic=traffic.get("bev_pool_op_bytes"),
                        ms=round(op_ms, 4), algorithmic_bytes=pool_bytes, peak_source=peaks["source"])
    roof_enc = dict(kernel="bevb200_encoder_forward: 21 x spconv_v6_kernel + rulebooks (side stream) + split + dense",
                    bound="tensor", achieved=round(enc_tflops, 3), peak=peaks["bf16_tflops_sustained"], unit="TFLOP/s",
                    frac=round(enc_tflops / peaks["bf16_tflops_sustained"], 5), traffic=traffic.get("encoder_bytes"),
                    ms=round(stages["encoder_ms"], 4), algorithmic_flops=flops, pairs=pairs, peak_source=peaks["source"],
                    note="useful FLOPs = sum 2*pairs*Cin*Cout over real (non-missing) neighbour pairs; the kernel issues "
                         "3 bf16 MMAs per fp32 product (BF16x3 split, 2 when the hi|lo weight images are merged) and also "
                         "multiplies the zero rows of missing neighbours")
    n_pts = int(pts.shape[0])
    vox_bytes = 4 * 5 * n_pts + n_vox * (4 * 5 + 16 + 4)        # points in; mean rows, (b,x,y,z), counts out
    vox_gbs = vox_bytes / (stages["voxelize_ms"] * 1e-3) / 1e9
    roof_vox = dict(kernel="hard_voxelize_mean (hash insert, lists, ballot scan, mean rows; fused, sync-free)", bound="hbm",
                    achieved=round(vox_gbs, 1), peak=peaks["hbm_gbs"], unit="GB/s", frac=round(vox_gbs / peaks["hbm_gbs"], 4),
                    traffic=None, ms=round(stages["voxelize_ms"], 4), algorithmic_bytes=vox_bytes,
                    points_per_s=round(n_pts / (stages["voxelize_ms"] * 1e-3)), peak_source=peaks["source"],
                    note="latency bound: ~9 MB of algorithmic traffic in ~8 dependent launches")
    # dominant kernel of the step: the tcgen05 sparse conv (21 launches per frame); each launch is timed alone
    # with CUDA events, achieved = useful FLOPs of those launches / their summed time (burst peak: timed alone)
    conv_ms, conv_launches, per_layer, conv_bwd_ms = conv_kernel_times(hp, pts, backward=True)
    conv_tflops = flops / (conv_ms * 1e-3) / 1e12
    roof_conv = dict(kernel="spconv_v6_kernel (tcgen05 SS-form implicit-GEMM sparse conv, BF16x3, pre-split operands; %d launches per frame)" % conv_launches,
                     bound="tensor", achieved=round(conv_tflops, 3), peak=peaks["bf16_tflops"], unit="TFLOP/s",
                     frac=round(conv_tflops / peaks["bf16_tflops"], 5), traffic=traffic.get("spconv_bytes"),
                     ms=round(conv_ms, 4), avg_launch_us=round(1e3 * conv_ms / max(conv_launches, 1), 2),
                     launches_per_frame=conv_launches, algorithmic_flops=flops, pairs=pairs, peak_source=peaks["source"],
                     traffic_source=traffic.get("source"), per_layer=per_layer,
                     note="achieved = sum over the frame's conv launches of 2*pairs*Cin*Cout (real neighbour pairs only) / "
                          "their summed CUDA-event time, each launch timed alone (burst bf16 peak as denominator); the "
                          "kernel issues 3 bf16 MMAs per fp32 product (hi/lo split) and also multiplies the zero rows of "
                          "missing neighbours, so the tensor pipe is busier than this fraction says")
    dominant = roof_conv if stages["encoder_ms"] >= stages["bev_pool_ms"] else roof_pool
    gpu_ref = None if args.no_gpu_reference else gpu_reference_leg(hp, x, pts)
    if gpu_ref and "frame_ms" in gpu_ref:
        ours_ms = stages["bev_pool_ms"] + stages["voxelize_ms"] + stages["encoder_ms"]
        gpu_ref["ours_frame_ms"] = round(ours_ms, 4)
        gpu_ref["speedup_frame"] = round(gpu_ref["frame_ms"] / ours_ms, 2)
        gpu_ref["speedup_bev_pool"] = round((gpu_ref["bev_pool_forward_ms"] + gpu_ref["bev_pool_sort_gather_ms"]) / stages["bev_pool_ms"], 2)
        gpu_ref["speedup_bev_pool_kernel_only"] = round(gpu_ref["bev_pool_forward_ms"] / op_ms, 2)
        gpu_ref["speedup_voxelize"] = round(gpu_ref["hard_voxelize_ms"] / stages["voxelize_ms"], 2)
        gpu_ref["speedup_encoder"] = round(gpu_ref["sparse_encoder_ms"] / stages["encoder_ms"], 2)
    del x
    torch.cuda.empty_cache()
    c5 = None if (args.no_c5 or world > 1) else c5_leg(device, peaks)
    # the CPU baseline is timed on rank 0 at N = 1 only
    cpu = None if (args.no_cpu_baseline or world > 1) else cpu_baseline(n_steps=1)
    line = {
        "metric": METRIC, "value": round(world * 1000.0 / ms_per_step, 3), "unit": "frames/s",
        "n_gpus": world, "steps": args.steps, "warmup": warm,
        "ms_per_step": round(ms_per_step, 4), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "frames_per_step_per_gpu": 1, "parallelism": "sample-parallel x%d" % world,
                   "launch": "the frame is one CUDA graph (no host synchronisation inside it: voxel and sparse-conv row "
                             "counts stay on the device), camera branch and LiDAR branch on two streams of the graph; "
                             "`eager` repeats it with python-issued launches; `stages_ms` times each stage alone",
                   "spconv_precision": {None: "bf16x3 (tcgen05 kind::f16, bf16 hi/lo split of fp32 operands, fp32 accumulate; default)",
                                        0: "fp32 (SIMT)", 1: "tf32x3", 2: "tf32", 3: "bf16x3"}[args.precision],
                   "l2": "inputs larger than L2: the 638 MB feature volume streams through L2 every step",
                   "bev_pool_plan": "rank/sort/interval tables cached per calibration (static geometry); see `bev_pool_prepare`",
                   "kept_rows": hp.n_kept, "intervals": hp.n_intervals, "numa_node": numa},
        "stages_ms": {k: round(v, 4) for k, v in stages.items()},
        "eager": {"value": round(world * 1000.0 / eager_ms, 3), "unit": "frames/s", "ms_per_step": round(eager_ms, 4),
                  "host_gap_ms": round(eager_ms - ms_per_step, 4)},
        "bev_pool_prepare": {"ms": round(prepare_ms, 4), "ms_from_geometry_tensor": round(prepare_geom_ms, 4),
                             "frames_per_s_plan_rebuilt_every_frame": round(world * 1000.0 / rebuild_ms, 3),
                             "ms_per_step_plan_rebuilt_every_frame": round(rebuild_ms, 4),
                             "note": "get_geometry fused into the plan build (from the calibration matrices) + quantise/filter/rank "
                                     "+ radix sort + interval tables of 1.99 M frustum points + one D2H count read (nuScenes camera2lidar is per sample: base.py:149-169, bev_pool.py:87-94 "
                                     "run every call in the reference)"},
        "e2e": {"value": round(world * 1000.0 / e2e_ms, 3), "unit": "frames/s", "ms_per_step": round(e2e_ms, 3),
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                "inputs": "pinned host: softmax depth [1,6,118,32,88] + context [1,6,32,88,80] (what the camera branch "
                          "hands the view transform, depth_lss.py:92-97) + points; outputs: both BEV maps to pinned host",
                "compute": "BEVPoolPlan.lift + voxelize + SparseEncoder captured once per input buffer set as a CUDA graph "
                           "(the API is sync-free) and replayed; H2D of frame i+1 / compute of frame i / D2H of frame i-1 on "
                           "three streams, every frame copies its inputs in and its results out"},
        "e2e_materialised": {"value": round(world * 1000.0 / e2e_mat_ms, 3), "unit": "frames/s",
                             "ms_per_step": round(e2e_mat_ms, 3), "h2d_bytes_per_step": h2d_mat,
                             "d2h_bytes_per_step": d2h, "steps": mat_steps,
                             "inputs": "pinned host: the materialised 638 MB lifted volume (drop-in bev_pool contract) + points"},
        "gpu_launches": int(launches),
        "bev_pool_extra": {"backward_ms": round(bwd_ms, 4), "backward_GBs": round(bwd_bytes / (bwd_ms * 1e-3) / 1e9, 1),
                           "backward_frac_of_hbm_peak": round(bwd_bytes / (bwd_ms * 1e-3) / 1e9 / peaks["hbm_gbs"], 4),
                           "fwd_plus_bwd_ms": round(pool_ms + bwd_ms, 4), "fused_lift_pool_ms": round(lift_ms, 4),
                           "fused_lift_pool_round1_row_kernel_ms": round(lift_rows_ms, 4),
                           "fused_lift_tables_build_ms_per_calibration": round(lift_prepare_ms, 3),
                           "note": "backward = bevpool_bwd_kernel through perm (660 MB algorithmic); fused lift+pool (column "
                                   "kernels): depth (8 MB) + ctx (5.4 MB) read once, per-segment rows written and read once, "
                                   "instead of one 320-byte context-row gather per kept point; graph-replay times"},
        "training": {"bev_pool_fwd_ms": round(pool_ms, 4), "bev_pool_bwd_ms": round(bwd_ms, 4),
                     "spconv_fwd_ms_21_convs": round(conv_ms, 4), "spconv_bwd_ms_21_convs": round(conv_bwd_ms, 4),
                     "note": "BASELINE config #2 asks for fwd+bwd: bev_pool backward = write stream through perm; spconv "
                             "backward per conv = input gradient (forward kernel on the transposed neighbour table, "
                             "bf16x3) + filter gradient (tensor cores: MN-major tcgen05 MMAs over the bf16 hi / lo "
                             "images, per-chunk partials + ordered reduction: bit-reproducible; spconv_wgrad_tc.cu); "
                             "each backward call timed alone"},
        "next_rows": next_rows,
        "roofline": dominant, "roofline_bev_pool": roof_pool, "roofline_bev_pool_op": roof_pool_op,
        "roofline_encoder": roof_enc, "roofline_voxelize": roof_vox,
        "gpu_reference": gpu_ref, "c4": c4, "c5": c5,
        "cpu_baseline": cpu, "clocks": clocks,
    }
    emit(line)


def hp_voxelize(pts, L):
    from bevfusion_b200.voxelize import Voxelization
    return Voxelization(L["voxel_size"], L["point_cloud_range"], L["max_num_points"], L["max_voxels"]).eval()(pts)


_REAL_STDOUT = None


def quiet_stdout():
    """Route fd 1 to stderr while the job runs (NCCL prints its version banner to stdout) so that
    stdout carries exactly ONE line: the JSON emitted by emit()."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the reference's CPU path on the host cores
# ---------------------------------------------------------------------------------------------
CPU_SAMPLE = ("per step: the WHOLE frame on the host cores -- bev_pool CPU path (torch QuickCumsum restatement, "
              "bev_pool.py:9-35 + base.py:149-169) on all 6 cameras (1.99 M x 80 rows), hard_voxelize C port on the full "
              "cloud, reference CPU spconv extension (oracle/_ref) SparseEncoder on the full voxel set; nothing extrapolated")


class CpuFrame:
    def __init__(self, seed=0):
        import oracle
        from oracle import reference_pipeline as RP
        from oracle.build_ref import built, load_ref
        from bevfusion_b200 import synthetic as S
        from bevfusion_b200.bev_pool import gen_dx_bx
        from bevfusion_b200.sparse_encoder import voxelnet_0p075_encoder
        self.oracle, self.RP, self.S = oracle, RP, S
        # the reference CPU path is small GEMMs + serial gather/scatter: it stops scaling (and then
        # regresses) beyond a few tens of threads, so use at most 16 of the host cores
        self.threads = min(os.cpu_count() or 1, 16)
        torch.set_num_threads(self.threads)
        self.kind = "reference" if built("sparse_conv_ext_ref") else "port"
        self.ref = load_ref("sparse_conv_ext_ref") if self.kind == "reference" else None
        self.geom, cfg = S.camera_geometry("C2")
        self.dx, self.bx, self.nx = gen_dx_bx(cfg["xbound"], cfg["ybound"], cfg["zbound"])
        g = torch.Generator().manual_seed(seed)
        block = torch.randn((118, 32, 88, 80), generator=g)
        self.x = torch.stack([block + 0.01 * cam for cam in range(6)]).unsqueeze(0)        # [1,6,118,32,88,80]
        self.points = S.lidar_cloud(seed=seed)
        torch.manual_seed(seed)
        self.encoder = voxelnet_0p075_encoder().eval()
        self.last = {}

    def step(self):
        """CPU seconds of one full frame (measured, not extrapolated)"""
        RP, L = self.RP, self.S.LIDAR_C3
        t0 = time.perf_counter()
        RP.bev_pool_cpu_quickcumsum(self.x, self.geom, self.dx, self.bx, self.nx)
        t1 = time.perf_counter()
        feats, coords = RP.voxelize_cpu(self.points, L, 160000)
        t2 = time.perf_counter()
        with torch.no_grad():
            if self.ref is not None:
                RP.reference_encoder_forward(self.ref, self.encoder, feats, coords, 1)
            else:
                self._port_encoder(feats, coords)
        t3 = time.perf_counter()
        self.last = {"bev_pool_s": round(t1 - t0, 3), "voxelize_s": round(t2 - t1, 3), "encoder_s": round(t3 - t2, 3)}
        return t3 - t0

    def _port_encoder(self, feats, coords):
        # oracle port of the first conv only (used when oracle/_ref is absent: then `kind` is "port" and the
        # encoder time is a lower bound)
        o = self.oracle
        w = self.encoder.conv_input[0].weight.detach().numpy()
        o.sparse_conv(feats.numpy(), coords.numpy(), 1, [1440, 1440, 41], w, [3, 3, 3], [1, 1, 1], [1, 1, 1],
                      [1, 1, 1], True, acc64=False)


def cpu_baseline(n_steps=1):
    cf = CpuFrame()
    secs = [cf.step() for _ in range(n_steps)]
    s = statistics.median(secs)
    return {"value": round(1.0 / s, 5), "unit": "frames/s", "cores": cf.threads, "kind": cf.kind,
            "sample": CPU_SAMPLE, "seconds_per_frame": round(s, 3), "stages": cf.last}


def run_reference(args, rank, world):
    """The reference's CPU implementation of the path on the host cores, whole frames.  A frame takes ~20 s, so
    the arm runs as many of the requested steps as fit a ~4 minute budget (at least one) and reports that
    count; warm-up is the construction of the inputs (no timed warm-up frame: nothing is cached between
    frames on this path)."""
    if rank != 0:
        return
    cf = CpuFrame()
    budget_s = float(os.environ.get("BEVB200_REFERENCE_BUDGET_S", "240"))
    secs = []
    t_start = time.perf_counter()
    while len(secs) < max(args.steps, 1):
        secs.append(cf.step())
        elapsed = time.perf_counter() - t_start
        if elapsed + max(secs) > budget_s:
            break
    s = sum(secs) / len(secs)
    value = round(1.0 / s, 5)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world,
            "steps": len(secs), "warmup": 0, "ms_per_step": round(s * 1000.0, 2),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "note": "CPU host cores only; one process regardless of n_gpus; whole frames "
                       "are timed (requested steps %d, run %d inside the %d s budget)" % (args.steps, len(secs), int(budget_s)),
                       "stages_s_last_frame": cf.last},
            "cpu_baseline": {"value": value, "unit": "frames/s", "cores": cf.threads, "kind": cf.kind,
                             "sample": CPU_SAMPLE},
            "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", type=int, default=None, help="spconv precision: 0 fp32, 1 tf32x3, 2 tf32, 3 bf16x3 (default)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU baseline leg (profiling runs)")
    ap.add_argument("--no-gpu-reference", action="store_true", help="skip the reference-CUDA-kernels leg")
    ap.add_argument("--no-c4", action="store_true", help="skip the full camera+LiDAR frame with the glue nets")
    ap.add_argument("--no-c5", action="store_true", help="skip the high-resolution stress configuration")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (float32, under 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    quiet_stdout()
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the hot path has no CPU fallback")
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout to the one JSON line
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
