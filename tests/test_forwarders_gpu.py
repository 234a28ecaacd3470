"""The drop-in boundary as CODE: integration/o3d_forwarders.cpp defines the reference's own `*CUDA` functions
(signatures from the reference's headers — RegistrationImpl.h:93-131, VoxelBlockGrid.h:345-381, Transform.h:42-47,
FixedRadiusIndex.h:227, 364 — compiled against them with the ref-shim's stub core::Tensor) as forwarders into
libo3db200.so.  integration/_build/libo3d_forwarders.so is built by integration/Makefile in the build container
(needs /root/reference) and travels to the GPU box.  CPU part: the library exports the reference's mangled
names.  GPU part: calling those functions gives the oracle's results.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

import oracle
from tests.synth import PRIMESENSE_K, camera_pose, make_colors, make_icp_pair, render_depth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "integration", "_build", "libo3d_forwarders.so")
needs_so = pytest.mark.skipif(not os.path.exists(SO), reason="integration/_build not built (needs the Open3D sources at build time)")

REFERENCE_SYMBOLS = [   # demangled prefixes the reference's callers link against
    "open3d::t::pipelines::kernel::ComputePosePointToPlaneCUDA(",
    "open3d::t::pipelines::kernel::ComputePoseColoredICPCUDA(",
    "open3d::t::geometry::kernel::transform::TransformPointsCUDA(",
    "open3d::t::geometry::kernel::transform::TransformNormalsCUDA(",
    "open3d::t::geometry::kernel::voxel_grid::DepthTouchCUDA(",
    "void open3d::t::geometry::kernel::voxel_grid::IntegrateCUDA<unsigned short, unsigned char, float, unsigned short, unsigned short>(",
    "void open3d::t::geometry::kernel::voxel_grid::IntegrateCUDA<unsigned short, unsigned char, float, float, float>(",
    "void open3d::t::geometry::kernel::voxel_grid::IntegrateCUDA<float, float, float, unsigned short, unsigned short>(",
    "void open3d::t::geometry::kernel::voxel_grid::IntegrateCUDA<float, float, float, float, float>(",
    "void open3d::core::nns::BuildSpatialHashTableCUDA<float>(",
    "void open3d::core::nns::HybridSearchCUDA<float, int>(",
]


@needs_so
def test_forwarder_library_exports_the_reference_symbols():
    out = subprocess.run(["nm", "-D", "-C", "--defined-only", SO], capture_output=True, text=True, check=True).stdout
    for sym in REFERENCE_SYMBOLS:
        assert sym in out, sym


def _lib():
    lib = C.CDLL(SO)
    lib.fwd_last_error.restype = C.c_char_p
    lib.fwd_depth_touch.restype = C.c_int64
    return lib


def _cuda(a, dtype=None):
    return torch.from_numpy(np.ascontiguousarray(a, dtype)).cuda()


def _p(t):
    return C.c_void_p(t.data_ptr())


def _d(a):
    return a.ctypes.data_as(C.c_void_p)


@needs_so
@pytest.mark.gpu
def test_compute_pose_point_to_plane_forwarder_vs_oracle():
    """ComputePosePointToPlaneCUDA through the reference's declaration: pose {6} f64 on the host, residual, count."""
    lib = _lib()
    src, tgt, nrm, _ = make_icp_pair(40000, seed=3)
    idx, _, _ = oracle.hybrid_search(tgt, src, 0.05, 1)
    corr = idx[:, 0].astype(np.int64)
    n = len(src)
    d = [_cuda(src), _cuda(tgt), _cuda(nrm), _cuda(corr)]
    pose, res, cnt = np.zeros(6), C.c_float(), C.c_int()
    for method, name, scale in ((0, "L2Loss", 1.0), (5, "TukeyLoss", 0.05)):
        rc = lib.fwd_compute_pose_point_to_plane(_p(d[0]), _p(d[1]), _p(d[2]), _p(d[3]), C.c_int64(n), method, C.c_double(scale),
                                                 C.c_double(1.0), _d(pose), C.byref(res), C.byref(cnt))
        assert rc == 0, lib.fwd_last_error()
        assert oracle.ROBUST[name] == method
        sums = oracle.pose_p2plane_sums(src, tgt, nrm, corr, robust=(name, scale, 1.0))
        ref_pose, ref_res, ref_cnt, singular = oracle.decode_and_solve_6x6(sums["sums64"])
        assert not singular and cnt.value == ref_cnt
        np.testing.assert_allclose(pose, ref_pose, rtol=2e-5, atol=1e-9)
        assert abs(res.value - ref_res) <= 1e-5 * abs(ref_res) + 1e-7


@needs_so
@pytest.mark.gpu
def test_transform_forwarders_vs_oracle():
    lib = _lib()
    src, _, nrm, T = make_icp_pair(5000, seed=4)
    nrm = nrm[: len(src)]
    p, q, Tg = _cuda(src), _cuda(nrm), _cuda(T, np.float32)
    assert lib.fwd_transform_points(_p(Tg), _p(p), _p(q), C.c_int64(len(src))) == 0, lib.fwd_last_error()
    T32 = T.astype(np.float32).astype(np.float64)
    # (same bar as test_icp_gpu.py::test_transform_points_and_normals: the stand-alone kernels may contract to FMAs)
    np.testing.assert_allclose(p.cpu().numpy(), oracle.transform_points(T32, src), rtol=2e-6, atol=2e-6)
    np.testing.assert_allclose(q.cpu().numpy(), oracle.transform_normals(T32, nrm), rtol=2e-6, atol=2e-6)


@needs_so
@pytest.mark.gpu
@pytest.mark.parametrize("f32_inputs,value_f32,color", [(False, False, True), (False, True, True), (True, False, True),
                                                         (True, True, True), (False, True, False)])
def test_depth_touch_and_integrate_forwarders_all_four_instantiations(f32_inputs, value_f32, color):
    """DepthTouchCUDA + IntegrateCUDA<in_depth, in_color, float, weight, color> on buffers laid out like the reference
    hash map's (keys [cap,3] i32, tsdf f32, weight / colour u16 or f32): block set and every voxel vs the oracle, 3
    frames.  Float32 weight / colour (the two instantiations round 1 lacked) go through the generic kernel."""
    lib = _lib()
    res, voxel, trunc, scale, dmax, cap = 16, 0.008, 0.064, 1000.0, 3.0, 3000
    K = np.ascontiguousarray(PRIMESENSE_K)
    keys = torch.zeros((cap, 3), dtype=torch.int32, device="cuda")
    tsdf = torch.zeros((cap, res ** 3), dtype=torch.float32, device="cuda")
    wdt = torch.float32 if value_f32 else torch.int16
    weight = torch.zeros((cap, res ** 3), dtype=wdt, device="cuda")
    cbuf = torch.zeros((cap, res ** 3, 3), dtype=wdt, device="cuda") if color else None
    okeys = np.zeros((cap, 3), np.int32)
    otsdf = np.zeros((cap, res ** 3), np.float32)
    owt = np.zeros((cap, res ** 3), np.float32 if value_f32 else np.uint16)
    ocol = np.zeros((cap, res ** 3, 3), np.float32 if value_f32 else np.uint16) if color else None
    size = 0
    for fid in (0, 30, 60):
        T = camera_pose(fid)
        E = np.ascontiguousarray(oracle.inverse_transformation(T))
        depth, col = render_depth(T, with_color=True)
        depth, col = depth.numpy(), col.numpy()
        if f32_inputs:
            depth, col = depth.astype(np.float32), col.astype(np.float32) / 255.0
        dg, cg = _cuda(depth), _cuda(col)
        coords = torch.zeros((cap, 3), dtype=torch.int32, device="cuda")
        n = lib.fwd_depth_touch(_p(dg), 0 if f32_inputs else 1, 480, 640, _d(K), _d(E), res, C.c_float(voxel), C.c_float(trunc),
                                C.c_float(scale), C.c_float(dmax), _p(coords), C.c_int64(cap))
        assert n > 0, lib.fwd_last_error()
        want = oracle.depth_touch(depth, PRIMESENSE_K, E, res, voxel, trunc, scale, dmax, 4)
        got = coords[:n].cpu().numpy()
        assert np.array_equal(got[np.lexsort((got[:, 2], got[:, 1], got[:, 0]))], want)
        # the reference's HashMap::Activate + Find (VoxelBlockGrid.cpp:313-315), played here by the oracle's map
        bi, _, size, rc = oracle.hashmap_activate(okeys, size, want)
        assert rc == 0
        keys[:size] = torch.from_numpy(okeys[:size]).cuda()
        big = _cuda(bi, np.int32)
        rc = lib.fwd_integrate(_p(dg), _p(cg) if color else None, 0 if f32_inputs else 1, 480, 640, _p(big), C.c_int64(len(bi)),
                               _p(keys), C.c_int64(cap), _p(tsdf), _p(weight), _p(cbuf) if color else None, 1 if value_f32 else 0,
                               _d(K), _d(K), _d(E), res, C.c_float(voxel), C.c_float(trunc), C.c_float(scale), C.c_float(dmax))
        assert rc == 0, lib.fwd_last_error()
        oracle.tsdf_integrate(depth, col if color else None, bi, okeys, otsdf, owt, ocol, PRIMESENSE_K, PRIMESENSE_K, E, res, voxel,
                              trunc, scale, dmax)
    gt, gw = tsdf.cpu().numpy(), weight.cpu().numpy()
    if not value_f32:
        gw = gw.view(np.uint16)
    assert np.array_equal(gw[:size], owt[:size]) and np.array_equal(gt[:size].view(np.uint32), otsdf[:size].view(np.uint32))
    if color:
        gc = cbuf.cpu().numpy()
        if not value_f32:
            gc = gc.view(np.uint16)
        assert np.array_equal(gc[:size], ocol[:size])
    assert int((gw[:size] > 0).sum()) > 100000


@needs_so
@pytest.mark.gpu
def test_hash_table_and_hybrid_search_forwarders_vs_oracle():
    lib = _lib()
    _, tgt, _, _ = make_icp_pair(20000, seed=6)
    rng = np.random.default_rng(0)
    q = (tgt[rng.integers(0, len(tgt), 5000)] + rng.normal(0, 0.01, (5000, 3))).astype(np.float32)
    r, k, H = 0.05, 4, max(len(tgt) // 32, 1)
    p, qg = _cuda(tgt), _cuda(q)
    tab = torch.zeros(len(tgt), dtype=torch.int32, device="cuda")
    splits = torch.zeros(H + 1, dtype=torch.int32, device="cuda")
    idx = torch.zeros((len(q), k), dtype=torch.int32, device="cuda")
    dist = torch.zeros((len(q), k), dtype=torch.float32, device="cuda")
    cnt = torch.zeros(len(q), dtype=torch.int32, device="cuda")
    rc = lib.fwd_hash_table_and_hybrid_search(_p(p), C.c_int64(len(tgt)), _p(qg), C.c_int64(len(q)), C.c_double(r), k, C.c_uint32(H),
                                              _p(tab), _p(splits), _p(idx), _p(dist), _p(cnt))
    assert rc == 0, lib.fwd_last_error()
    oi, od, oc = oracle.hybrid_search(tgt, q, r, k)
    assert np.array_equal(idx.cpu().numpy(), oi) and np.array_equal(cnt.cpu().numpy(), oc)
    assert np.array_equal(dist.cpu().numpy().view(np.uint32), od.view(np.uint32))
    sp = splits.cpu().numpy().view(np.uint32)
    assert sp[0] == 0 and sp[-1] == len(tgt) and (np.diff(sp.astype(np.int64)) >= 0).all()
    assert np.array_equal(np.sort(tab.cpu().numpy()), np.arange(len(tgt)))
