#!/usr/bin/env python
"""Record what the reference's own code returns on the inputs of tests/test_oracle_vs_ref*.py into
tests/golden/ref_oracle_vs_ref.npz and tests/golden/ref_oracle_vs_ref_vbg.npz.

Needs oracle/_ref/libo3dref.so, which build() compiles from the Open3D sources (oracle/ref_shim) where they are
present; the tests themselves only read the stored arrays.  Run from the repository root after build():

    python tests/golden/make_ref_vectors.py
"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import oracle  # noqa: E402
from tests import test_oracle_vs_ref as T  # noqa: E402
from tests import test_oracle_vs_ref_vbg as V  # noqa: E402
from tests.ref_vectors import GOLDEN, pack  # noqa: E402
from tests.synth import PRIMESENSE_K, camera_pose  # noqa: E402

REF = os.path.join(ROOT, "oracle", "_ref", "libo3dref.so")
f32p, f64p, i64p, i32p = (C.POINTER(t) for t in (C.c_float, C.c_double, C.c_int64, C.c_int))
vp = C.c_void_p


def _p(a, t):
    return a.ctypes.data_as(t)


def load_ref():
    L = C.CDLL(REF)
    L.ref_spatial_hash.restype = C.c_uint64
    L.ref_spatial_hash.argtypes = [C.c_int] * 3
    L.ref_minivec_hash_i32x3.restype = C.c_uint64
    L.ref_minivec_hash_i32x3.argtypes = [C.c_int] * 3
    L.ref_robust_weight_f64.restype = C.c_double
    L.ref_robust_weight_f64.argtypes = [C.c_int, C.c_double, C.c_double, C.c_double]
    L.ref_robust_weight_f32.restype = C.c_float
    L.ref_robust_weight_f32.argtypes = [C.c_int, C.c_double, C.c_double, C.c_float]
    L.ref_jacobian_p2plane_f32.argtypes = [C.c_int64, f32p, f32p, f32p, i64p, f32p, f32p]
    L.ref_jacobian_colored_f32.argtypes = [C.c_int64] + [f32p] * 6 + [i64p, C.c_float, C.c_float, f32p, f32p, f32p, f32p]
    L.ref_pose_to_transformation.argtypes = [f64p, f64p]
    L.ref_transform_points_f32.argtypes = [f32p, f32p, C.c_int64]
    L.ref_transform_normals_f32.argtypes = [f32p, f32p, C.c_int64]
    L.ref_compute_voxel_index_f32.argtypes = [f32p, C.c_float, i32p]
    L.ref_transform_indexer.argtypes = [f64p, f64p, C.c_float, C.c_int, f32p, f32p]
    L.ref_workload_to_coord3.argtypes = [C.c_int, C.c_int, i32p]
    L.ref_in_boundary2.argtypes = [C.c_int, C.c_int, C.c_float, C.c_float]
    L.ref_solve_svd3x3_f32.argtypes = [f32p, f32p, f32p]
    L.ref_clip_transform.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float, f32p]
    L.ref_pyr_down_depth.argtypes = [f32p, C.c_int, C.c_int, C.c_float, C.c_float, f32p]
    L.ref_create_vertex_map.argtypes = [f32p, C.c_int, C.c_int, f64p, C.c_float, f32p]
    L.ref_create_normal_map.argtypes = [f32p, C.c_int, C.c_int, C.c_float, f32p]
    L.ref_huber_deriv.restype = C.c_float
    L.ref_huber_deriv.argtypes = [C.c_float, C.c_float]
    L.ref_huber_loss.restype = C.c_float
    L.ref_huber_loss.argtypes = [C.c_float, C.c_float]
    L.ref_odometry_jacobian_p2plane.argtypes = [C.c_int, C.c_int, C.c_float, f32p, f32p, f32p, C.c_int, C.c_int,
                                                f64p, f64p, f32p, f32p]
    L.ref_pose_p2plane_sums_f32.argtypes = [f32p, f32p, f32p, i64p, C.c_int64, C.c_int64, C.c_int, C.c_double,
                                            C.c_double, f64p]
    L.ref_pose_colored_sums_f32.argtypes = [f32p] * 6 + [i64p, C.c_int64, C.c_int64, C.c_int, C.c_double, C.c_double,
                                                         C.c_double, f64p]
    L.ref_odometry_p2plane_sums.argtypes = [f32p, f32p, f32p, C.c_int, C.c_int, f64p, f64p, C.c_float, C.c_float, f64p]
    L.ref_color_gradient_point_f32.argtypes = [f32p, f32p, f32p, C.c_int64, i32p, C.c_int32, f32p]
    L.ref_information_matrix_f32.argtypes = [f32p, C.c_int64, i64p, C.c_int64, f64p]
    L.ref_depth_touch.restype = C.c_int64
    L.ref_depth_touch.argtypes = [vp, C.c_int, C.c_int, C.c_int, f64p, f64p, C.c_int, C.c_float, C.c_float, C.c_float,
                                  C.c_float, C.c_int, i32p, C.c_int64]
    L.ref_integrate_f32_values.restype = None
    L.ref_integrate_f32_values.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, i32p, C.c_int64, i32p, C.c_int64, f32p, vp,
                                           vp, f64p, f64p, f64p, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float]
    L.ref_integrate.restype = None
    L.ref_integrate.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, i32p, C.c_int64, i32p, C.c_int64, f32p, vp, vp, f64p,
                                f64p, f64p, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float]
    L.ref_estimate_range.restype = C.c_int64
    L.ref_estimate_range.argtypes = [i32p, C.c_int64, f64p, f64p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float,
                                     C.c_float, C.c_float, C.c_int64, f32p]
    L.ref_ray_cast.restype = None
    L.ref_ray_cast.argtypes = [i32p, C.c_int64, f32p, vp, vp, f32p, f64p, f64p, C.c_int, C.c_int, C.c_int, C.c_float,
                               C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int] + [vp] * 10
    return L


def _sums_f32_from_jacobians(ref, src, tgt, nrm, corr):
    """The 29 point-to-plane sums accumulated in f32, in index order, from the reference's Jacobian function."""
    acc = np.zeros(29, np.float32)
    J = np.zeros(6, np.float32)
    r = C.c_float(0)
    for i in range(len(src)):
        if not ref.ref_jacobian_p2plane_f32(i, _p(src, f32p), _p(tgt, f32p), _p(nrm, f32p), _p(corr, i64p), _p(J, f32p),
                                            C.byref(r)):
            continue
        rr = np.float32(r.value)
        s = 0
        for j in range(6):
            for k in range(j + 1):
                acc[s] += J[j] * np.float32(1.0) * J[k]
                s += 1
            acc[21 + j] += J[j] * np.float32(1.0) * rr
        acc[27] += rr
        acc[28] += np.float32(1)
    return acc


def _colored_sums_from_jacobians(ref, src, sc, tgt, nrm, tc, grad, corr, lam):
    slg, slp = np.float32(np.sqrt(lam)), np.float32(np.sqrt(1.0 - lam))
    acc = np.zeros(29, np.float64)
    JG, JI = np.zeros(6, np.float32), np.zeros(6, np.float32)
    rG, rI = C.c_float(0), C.c_float(0)
    one = np.float32(1)
    for i in range(len(src)):
        ok = ref.ref_jacobian_colored_f32(i, _p(src, f32p), _p(sc, f32p), _p(tgt, f32p), _p(nrm, f32p), _p(tc, f32p),
                                          _p(grad, f32p), _p(corr, i64p), float(slg), float(slp), _p(JG, f32p),
                                          _p(JI, f32p), C.byref(rG), C.byref(rI))
        if not ok:
            continue
        g, q = np.float32(rG.value), np.float32(rI.value)
        s = 0
        for j in range(6):
            for k in range(j + 1):
                acc[s] += np.float32(JG[j] * one * JG[k] + JI[j] * one * JI[k])
                s += 1
            acc[21 + j] += np.float32(JG[j] * one * g + JI[j] * one * q)
        acc[27] += np.float32(g * g + q * q)
        acc[28] += 1
    return acc


def record_oracle_vs_ref(ref):
    out = {}
    keys, cells, points = T.hash_inputs()
    pack(out, "minivec_hash", np.array([ref.ref_minivec_hash_i32x3(*map(int, k)) for k in keys], np.uint64))
    pack(out, "spatial_hash", np.array([ref.ref_spatial_hash(*map(int, c)) for c in cells], np.uint64))
    vox = np.zeros((len(points), 3), np.int32)
    for i, (p, inv) in enumerate(points):
        a = np.array(p, np.float32)
        ref.ref_compute_voxel_index_f32(_p(a, f32p), inv, _p(vox[i], i32p))
    pack(out, "voxel_index", vox)

    shape = (7, len(T.ROBUST_SCALES), len(T.ROBUST_SHAPES), len(T.ROBUST_RS))
    w64, w32 = np.zeros(shape), np.zeros(shape, np.float32)
    for idx in np.ndindex(*shape):
        m, i, j, k = idx
        args = (m, T.ROBUST_SCALES[i], T.ROBUST_SHAPES[j], T.ROBUST_RS[k])
        w64[idx], w32[idx] = ref.ref_robust_weight_f64(*args), ref.ref_robust_weight_f32(*args)
    pack(out, "robust_weight_f64", w64)
    pack(out, "robust_weight_f32", w32)

    pack(out, "p2plane_jacobian_sums32", _sums_f32_from_jacobians(ref, *T.p2plane_inputs()))
    pack(out, "colored_jacobian_sums64", _colored_sums_from_jacobians(ref, *T.colored_inputs()))

    poses, Tm, pts = T.pose_inputs()
    Ts = np.zeros((len(poses), 16))
    for i, pose in enumerate(poses):
        pose = np.ascontiguousarray(pose)
        ref.ref_pose_to_transformation(_p(pose, f64p), _p(Ts[i], f64p))
    pack(out, "pose_to_transformation", Ts)
    Tf = np.ascontiguousarray(Tm.astype(np.float32))
    a, b = pts.copy(), pts.copy()
    ref.ref_transform_points_f32(_p(Tf, f32p), _p(a, f32p), len(a))
    ref.ref_transform_normals_f32(_p(Tf, f32p), _p(b, f32p), len(b))
    pack(out, "transform_points", a)
    pack(out, "transform_normals", b)
    coords = []
    for res in (2, 8, 16):
        for w in range(0, res ** 3, 7):
            c3 = np.zeros(3, np.int32)
            ref.ref_workload_to_coord3(res, w, _p(c3, i32p))
            coords.append(c3)
    pack(out, "workload_to_coord3", np.array(coords, np.int32))
    pack(out, "in_boundary2", np.array([bool(ref.ref_in_boundary2(480, 640, x, y)) for x, y in T.BOUNDARY_POINTS]))

    K, E, _, _, _, samples = T.tsdf_geometry_inputs()
    cams, uvs = np.zeros((len(samples), 3), np.float32), np.zeros((len(samples), 3), np.float32)
    for i, (_, _, vin) in enumerate(samples):
        ref.ref_transform_indexer(_p(K, f64p), _p(E, f64p), 0.008, 0, _p(vin, f32p), _p(cams[i], f32p))
        ref.ref_transform_indexer(_p(K, f64p), _p(E, f64p), 0.008, 1, _p(cams[i], f32p), _p(uvs[i], f32p))
    pack(out, "indexer_cam", cams)
    pack(out, "indexer_uv", uvs)
    pack(out, "indexer_in_boundary", np.array([bool(ref.ref_in_boundary2(480, 640, float(u[0]), float(u[1])))
                                               for u in uvs]))

    x = []
    for _, A32, b32 in T.svd3_systems():
        want = np.zeros(3, np.float32)
        ref.ref_solve_svd3x3_f32(_p(A32, f32p), _p(b32, f32p), _p(want, f32p))
        x.append(want)
    pack(out, "solve_svd3x3_f32", np.array(x))
    x = []
    for A, b in T.gradient_like_systems():
        A32, b32, x32 = A.ravel().astype(np.float32), b.astype(np.float32), np.zeros(3, np.float32)
        ref.ref_solve_svd3x3_f32(_p(A32, f32p), _p(b32, f32p), _p(x32, f32p))
        x.append(x32)
    pack(out, "gradient_like_solve_svd3x3_f32", np.array(x))

    da, _, _, K = T.odometry_inputs()
    rows, cols = da.shape
    nan = float("nan")
    for src, is_f32 in ((da, 0), ((da.astype(np.float32) / 1000.0), 1)):
        src = np.ascontiguousarray(src)
        want = np.empty((rows, cols), np.float32)
        scale = 1000.0 if not is_f32 else 1.0
        ref.ref_clip_transform(src.ctypes.data, is_f32, rows, cols, scale, 0.0, 3.0, nan, _p(want, f32p))
        pack(out, f"clip_transform_{is_f32}", want)
    depth = oracle.clip_transform(da)
    r, c = rows, cols
    Kp = K.copy()
    for level in range(3):
        v = np.empty((r, c, 3), np.float32)
        ref.ref_create_vertex_map(_p(depth, f32p), r, c, _p(np.ascontiguousarray(Kp.reshape(9)), f64p), nan, _p(v, f32p))
        n = np.empty((r, c, 3), np.float32)
        ref.ref_create_normal_map(_p(v, f32p), r, c, nan, _p(n, f32p))
        d = np.empty((r // 2, c // 2), np.float32)
        ref.ref_pyr_down_depth(_p(depth, f32p), r, c, 0.14, nan, _p(d, f32p))
        pack(out, f"vertex_map_{level}", v)
        pack(out, f"normal_map_{level}", n)
        pack(out, f"pyr_down_depth_{level}", d)
        depth = d
        r, c = r // 2, c // 2
        Kp = Kp / 2
        Kp[2, 2] = 1
    d0 = np.where(np.isnan(oracle.clip_transform(da)), np.float32(0), oracle.clip_transform(da))
    v = np.empty((rows, cols, 3), np.float32)
    ref.ref_create_vertex_map(_p(d0, f32p), rows, cols, _p(np.ascontiguousarray(K.reshape(9)), f64p), 0.0, _p(v, f32p))
    n = np.empty((rows, cols, 3), np.float32)
    ref.ref_create_normal_map(_p(v, f32p), rows, cols, 0.0, _p(n, f32p))
    d = np.empty((rows // 2, cols // 2), np.float32)
    ref.ref_pyr_down_depth(_p(d0, f32p), rows, cols, 0.14, 0.0, _p(d, f32p))
    pack(out, "vertex_map_fill0", v)
    pack(out, "normal_map_fill0", n)
    pack(out, "pyr_down_depth_fill0", d)

    rs = T.huber_residuals()
    pack(out, "huber_deriv", np.float32([[ref.ref_huber_deriv(r, d) for d in T.HUBER_DELTAS] for r in rs]))
    pack(out, "huber_loss", np.float32([[ref.ref_huber_loss(r, d) for d in T.HUBER_DELTAS] for r in rs]))
    sv, tv, tn, Kp, Tp = T.odometry_level(2)
    rows, cols = sv.shape[:2]
    Kf, Tf = np.ascontiguousarray(Kp.reshape(9)), np.ascontiguousarray(Tp.reshape(16))
    ok = np.zeros((rows, cols), bool)
    Jall, rall = np.zeros((rows, cols, 6), np.float32), np.zeros((rows, cols), np.float32)
    J, r = np.zeros(6, np.float32), np.zeros(1, np.float32)
    for y in range(rows):
        for x in range(cols):
            ok[y, x] = ref.ref_odometry_jacobian_p2plane(x, y, 0.07, _p(sv, f32p), _p(tv, f32p), _p(tn, f32p), rows, cols,
                                                         _p(Kf, f64p), _p(Tf, f64p), _p(J, f32p), _p(r, f32p))
            if ok[y, x]:
                Jall[y, x], rall[y, x] = J, r[0]
    pack(out, "odometry_jacobian_valid", ok)
    pack(out, "odometry_jacobian_J", Jall)
    pack(out, "odometry_jacobian_r", rall)

    from tests.synth import make_colors, make_icp_pair
    src, tgt, nrm, _ = make_icp_pair(6000, seed=12)
    idx, _, _ = oracle.hybrid_search(tgt, src, 0.05, 1)
    corr = np.ascontiguousarray(idx[:, 0].astype(np.int64))
    sc, tc = make_colors(src, 1), make_colors(tgt, 1)
    grad = np.ascontiguousarray(np.random.default_rng(1).normal(0, 0.5, tgt.shape).astype(np.float32))
    for name, scale, shape in T.ROBUST:
        method = oracle.ROBUST[name]
        want = np.zeros(29)
        ref.ref_pose_p2plane_sums_f32(_p(src, f32p), _p(tgt, f32p), _p(nrm, f32p), _p(corr, i64p), len(src), len(tgt),
                                      method, scale, shape, _p(want, f64p))
        pack(out, f"pose_p2plane_sums_{name}", want.copy())
        ref.ref_pose_colored_sums_f32(_p(src, f32p), _p(sc, f32p), _p(tgt, f32p), _p(nrm, f32p), _p(tc, f32p),
                                      _p(grad, f32p), _p(corr, i64p), len(src), len(tgt), method, scale, shape, 0.968,
                                      _p(want, f64p))
        pack(out, f"pose_colored_sums_{name}", want.copy())

    sv, tv, tn, Kp, Tp = T.odometry_level(1)
    want = np.zeros(29)
    Kf, Tf = np.ascontiguousarray(Kp.reshape(9)), np.ascontiguousarray(Tp.reshape(16))
    ref.ref_odometry_p2plane_sums(_p(sv, f32p), _p(tv, f32p), _p(tn, f32p), sv.shape[0], sv.shape[1], _p(Kf, f64p),
                                  _p(Tf, f64p), 0.07, 0.05, _p(want, f64p))
    pack(out, "odometry_p2plane_sums", want)

    grads = []
    for _, pts, nrm, col in T.color_gradient_clusters():
        idx, _, cnt = oracle.hybrid_search(pts, pts, 10.0, 30)
        want = np.full_like(pts, 7.0)
        for i in range(len(pts)):
            row = np.ascontiguousarray(idx[i], np.int32)
            ref.ref_color_gradient_point_f32(_p(pts, f32p), _p(nrm, f32p), _p(col, f32p), i, _p(row, i32p), int(cnt[i]),
                                             _p(want, f32p))
        grads.append(want)
    pack(out, "color_gradients", np.concatenate(grads))
    pts, nrm, col = T.tiny_cluster()
    want = np.full_like(pts, 7.0)
    row = np.int32([0, 1, 2])
    ref.ref_color_gradient_point_f32(_p(pts, f32p), _p(nrm, f32p), _p(col, f32p), 0, _p(row, i32p), 3, _p(want, f32p))
    pack(out, "color_gradient_three_neighbours", want[0])

    tgt, corr = T.information_matrix_inputs()
    want = np.zeros(36)
    ref.ref_information_matrix_f32(_p(tgt, f32p), len(tgt), _p(corr, i64p), len(corr), _p(want, f64p))
    pack(out, "information_matrix", want)
    return out


def record_oracle_vs_ref_vbg(ref):
    RES, VOXEL, TRUNC, SCALE, DMIN, DMAX = V.RES, V.VOXEL, V.TRUNC, V.SCALE, V.DMIN, V.DMAX
    K9 = V.K9
    out = {}
    for fid, f32 in V.DEPTH_TOUCH_FRAMES:
        E, depth, _ = V.frame(fid, f32)
        Ef = np.ascontiguousarray(E.reshape(16))
        buf = np.zeros((76800, 3), np.int32)
        n = ref.ref_depth_touch(depth.ctypes.data, int(f32), 480, 640, _p(K9, f64p), _p(Ef, f64p), RES, VOXEL,
                                VOXEL * TRUNC, SCALE, DMAX, 4, _p(buf, i32p), len(buf))
        pack(out, f"depth_touch_{fid}_{int(f32)}", V.sorted_keys(buf[:n]))

    def integrate(fn, steps, cap, value_dtype, f32_inputs, with_color=True):
        """The reference's IntegrateCPU into its own buffers, on the block indices the oracle's hash map assigns."""
        keys = np.zeros((cap, 3), np.int32)
        t = np.zeros((cap, RES ** 3), np.float32)
        w = np.zeros((cap, RES ** 3), value_dtype)
        col = np.zeros((cap, RES ** 3, 3), value_dtype)
        size = 0
        for fid in steps:
            E, depth, color = V.frame(fid, f32_inputs)
            touched = oracle.depth_touch(depth, PRIMESENSE_K, E, RES, VOXEL, VOXEL * TRUNC, SCALE, DMAX, 4)
            bi, _, size, _ = oracle.hashmap_activate(keys, size, touched)
            Ef = np.ascontiguousarray(E.reshape(16))
            bi = np.ascontiguousarray(bi, np.int32)
            fn(depth.ctypes.data, color.ctypes.data if with_color else None, int(f32_inputs), 480, 640, _p(bi, i32p),
               len(bi), _p(keys, i32p), cap, _p(t, f32p), w.ctypes.data, col.ctypes.data if with_color else None,
               _p(K9, f64p), _p(K9, f64p), _p(Ef, f64p), RES, VOXEL, VOXEL * TRUNC, SCALE, DMAX)
        return t, w, col

    t, w, col = integrate(ref.ref_integrate, V.VOLUME_FRAMES, V.VOLUME_CAPACITY, np.uint16, False)
    pack(out, "integrate_tsdf", t)
    pack(out, "integrate_weight", w)
    pack(out, "integrate_color", col)
    for with_color in (True, False):
        t, w, col = integrate(ref.ref_integrate, (300,), 3000, np.uint16, True, with_color)
        pack(out, f"integrate_f32_inputs_{int(with_color)}_tsdf", t)
        pack(out, f"integrate_f32_inputs_{int(with_color)}_weight", w)
        pack(out, f"integrate_f32_inputs_{int(with_color)}_color", col)
    for f32_inputs in (False, True):
        t, w, col = integrate(ref.ref_integrate_f32_values, (300, 302, 304), 3000, np.float32, f32_inputs)
        pack(out, f"integrate_f32_values_{int(f32_inputs)}_tsdf", t)
        pack(out, f"integrate_f32_values_{int(f32_inputs)}_weight", w)
        pack(out, f"integrate_f32_values_{int(f32_inputs)}_color", col)

    vol = V.oracle_volume()
    E = oracle.inverse_transformation(camera_pose(V.VOLUME_FRAMES[-1]))
    Ef = np.ascontiguousarray(E.reshape(16))
    keys = np.ascontiguousarray(vol["frustum"])
    for down in V.RANGE_DOWN:
        want = np.zeros((480 // down, 640 // down, 2), np.float32)
        for name, fragments in (("", 1 << 16), ("_auto", 0), ("_small", 40)):
            rng = np.zeros_like(want)
            n = ref.ref_estimate_range(_p(keys, i32p), len(keys), _p(K9, f64p), _p(Ef, f64p), 480, 640, down, RES, VOXEL,
                                       DMIN, DMAX, fragments, _p(rng, f32p))
            if name == "_small":                # stored whole: the test counts its valid cells
                out[f"estimate_range_{down}{name}"] = rng
            else:
                pack(out, f"estimate_range_{down}{name}", rng)
            if name == "_auto":
                pack(out, f"estimate_range_{down}_auto_fragments", np.int64(n))

    okeys = np.ascontiguousarray(vol["keys"])
    o = vol["o"]
    for fid, threshold in V.RAY_CAST_VIEWS:
        E = oracle.inverse_transformation(camera_pose(fid))
        Ef = np.ascontiguousarray(E.reshape(16))
        rng = oracle.estimate_range(okeys[: vol["size"]], PRIMESENSE_K, E, 480, 640, 8, RES, VOXEL, DMIN, DMAX)
        want = {}
        for name in V.RAY_CAST_ATTRS:
            c, dt = oracle.RAYCAST_ATTRS[name]
            want[name] = np.full((480, 640, c), 77, dt)
        ref.ref_ray_cast(_p(okeys, i32p), vol["size"], _p(o["tsdf"], f32p), o["wt"].ctypes.data, o["col"].ctypes.data,
                         _p(rng, f32p), _p(K9, f64p), _p(Ef, f64p), 480, 640, RES, VOXEL, SCALE, DMIN, DMAX, threshold,
                         TRUNC, 8, *[want[name].ctypes.data for name in V.RAY_CAST_ATTRS])
        for name in V.RAY_CAST_ATTRS:
            pack(out, f"ray_cast_{fid}_{name}", want[name].astype(bool) if name == "mask" else want[name])
    return out


def main():
    if not os.path.exists(REF):
        raise SystemExit(f"{REF} not found: build() compiles it where the Open3D sources are present")
    ref = load_ref()
    for module, record in (("oracle_vs_ref", record_oracle_vs_ref), ("oracle_vs_ref_vbg", record_oracle_vs_ref_vbg)):
        path = os.path.join(GOLDEN, f"ref_{module}.npz")
        np.savez_compressed(path, **record(ref))
        print(f"wrote {path} ({os.path.getsize(path)} bytes)")


if __name__ == "__main__":
    main()
