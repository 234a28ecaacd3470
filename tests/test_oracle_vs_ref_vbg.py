"""The oracle's voxel-block-grid path against the reference's OWN CPU implementation: t/geometry/kernel/
VoxelBlockGridCPU.cpp + VoxelBlockGridImpl.h compiled unmodified (oracle/ref_shim/ref_shim_vbg.cpp, stub
Tensor/HashMap/TBB headers, serial ParallelFor): what DepthTouchCPU, IntegrateCPU, EstimateRangeCPU and RayCastCPU
return on the inputs built here, stored in tests/golden/ref_oracle_vs_ref_vbg.npz by tests/golden/make_ref_vectors.py.
Every comparison is bit-exact.  CPU only."""
import functools

import numpy as np
import pytest

import oracle
from tests.ref_vectors import Vectors
from tests.synth import PRIMESENSE_K, camera_pose, render_depth

VOXEL, RES, TRUNC = 0.008, 16, 8.0
SCALE, DMIN, DMAX = 1000.0, 0.1, 3.0
K9 = np.ascontiguousarray(np.asarray(PRIMESENSE_K, np.float64).reshape(9))
DEPTH_TOUCH_FRAMES = [(0, False), (137, False), (500, True)]
VOLUME_FRAMES, VOLUME_CAPACITY = (100, 102, 104, 106), 4000
RANGE_DOWN = [8, 4]
RAY_CAST_VIEWS = [(106, 3.0), (103, 1.0), (140, 1.0)]
RAY_CAST_ATTRS = ("depth", "vertex", "color", "normal", "index", "mask", "interp_ratio", "interp_ratio_dx",
                  "interp_ratio_dy", "interp_ratio_dz")


@pytest.fixture(scope="module")
def ref():
    return Vectors("oracle_vs_ref_vbg")


def frame(i, f32=False):
    T = camera_pose(i)
    depth, color = render_depth(T, with_color=True)
    depth, color = depth.numpy(), color.numpy()
    if f32:
        depth, color = depth.astype(np.float32), color.astype(np.float32) / 255.0
    return oracle.inverse_transformation(T), np.ascontiguousarray(depth), np.ascontiguousarray(color)


def sorted_keys(k):
    k = np.asarray(k, np.int32).reshape(-1, 3)
    return k[np.lexsort((k[:, 2], k[:, 1], k[:, 0]))]


def fuse(frames, cap, value_dtype=np.uint16, f32_inputs=False, with_color=True):
    """`frames` fused by the oracle: the hash map's keys and size, tsdf / weight / colour buffers, last frustum."""
    keys = np.zeros((cap, 3), np.int32)
    t, w = np.zeros((cap, RES ** 3), np.float32), np.zeros((cap, RES ** 3), value_dtype)
    col = np.zeros((cap, RES ** 3, 3), value_dtype)
    size, touched = 0, None
    for fid in frames:
        E, depth, color = frame(fid, f32_inputs)
        touched = oracle.depth_touch(depth, PRIMESENSE_K, E, RES, VOXEL, VOXEL * TRUNC, SCALE, DMAX, 4)
        bi, _, size, rc = oracle.hashmap_activate(keys, size, touched)
        assert rc == 0
        oracle.tsdf_integrate(depth, color if with_color else None, bi, keys, t, w, col if with_color else None,
                              PRIMESENSE_K, PRIMESENSE_K, E, RES, VOXEL, VOXEL * TRUNC, SCALE, DMAX)
    return dict(keys=keys, size=size, o=dict(tsdf=t, wt=w, col=col), frustum=touched)


@functools.lru_cache(maxsize=1)
def oracle_volume():
    """Four colour frames fused by the oracle (the reference's IntegrateCPU fuses the same frames on the same block
    indices into the stored buffers)."""
    return fuse(VOLUME_FRAMES, VOLUME_CAPACITY)


@pytest.mark.parametrize("fid,f32", DEPTH_TOUCH_FRAMES)
def test_depth_touch_is_the_reference_block_set(ref, fid, f32):
    """DepthTouchCPU (VoxelBlockGridCPU.cpp:117-201): identical set of touched blocks."""
    E, depth, _ = frame(fid, f32)
    got = oracle.depth_touch(depth, PRIMESENSE_K, E, RES, VOXEL, VOXEL * TRUNC, SCALE, DMAX, 4)
    assert len(got) > 300
    ref.check(f"depth_touch_{fid}_{int(f32)}", np.asarray(got, np.int32))


def test_integrate_is_the_reference_integrate(ref):
    """IntegrateCPU<u16,u8,f32,u16,u16> (VoxelBlockGridImpl.h:151-308) over 4 frames: tsdf bit for bit, weights and
    colours equal."""
    o = oracle_volume()["o"]
    assert (o["wt"] > 0).sum() > 500000
    ref.check("integrate_weight", o["wt"])
    ref.check("integrate_color", o["col"])
    ref.check("integrate_tsdf", o["tsdf"])


def test_integrate_float_inputs_and_depth_only(ref):
    """IntegrateCPU<f32,f32,f32,u16,u16> (colour x 255) and the depth-only call (empty colour tensor)."""
    for with_color in (True, False):
        o = fuse((300,), 3000, f32_inputs=True, with_color=with_color)["o"]
        for name, key in (("tsdf", "tsdf"), ("weight", "wt"), ("color", "col")):
            ref.check(f"integrate_f32_inputs_{int(with_color)}_{name}", o[key])
        assert o["col"].any() == with_color


@pytest.mark.parametrize("f32_inputs", [False, True])
def test_integrate_float32_value_layout_is_the_reference_integrate(ref, f32_inputs):
    """The reference's other value layout — IntegrateCPU<u16,u8,f32,float,float> and <f32,f32,f32,float,float>
    (weight Float32, colour Float32, VoxelBlockGridCPU.cpp instantiations) — over 3 fused frames: tsdf, weight and
    colour bit for bit (the float colour is NOT truncated to an integer in this layout)."""
    o = fuse((300, 302, 304), 3000, np.float32, f32_inputs)["o"]
    for name, key in (("tsdf", "tsdf"), ("weight", "wt"), ("color", "col")):
        ref.check(f"integrate_f32_values_{int(f32_inputs)}_{name}", o[key])
    assert o["wt"].max() == 3.0 and (o["col"] != np.floor(o["col"])).any()


@pytest.mark.parametrize("down", RANGE_DOWN)
def test_estimate_range_is_the_reference_range_map(ref, down):
    """EstimateRangeCPU (VoxelBlockGridImpl.h:310-555) with a fragment buffer that is large enough; and what upstream
    does when it is not (the mode this library does not have)."""
    vol = oracle_volume()
    E = oracle.inverse_transformation(camera_pose(VOLUME_FRAMES[-1]))
    got = oracle.estimate_range(np.ascontiguousarray(vol["frustum"]), PRIMESENSE_K, E, 480, 640, down, RES, VOXEL,
                                DMIN, DMAX)
    assert (got[..., 0] < got[..., 1]).mean() > 0.9
    ref.check(f"estimate_range_{down}", got)
    # upstream's own first-call allocation, h_down*w_down/256/voxel_size fragments (:341-347) ...
    assert ref[f"estimate_range_{down}_auto_fragments"] >= (480 // down) * (640 // down) // 256 / VOXEL - 1
    ref.check(f"estimate_range_{down}_auto", got)
    # ... and a buffer that is too small: fragments are dropped, the map is incomplete (warning upstream)
    small = ref[f"estimate_range_{down}_small"]
    assert not np.array_equal(small, got) and ((small[..., 0] < small[..., 1]).sum() < (got[..., 0] < got[..., 1]).sum())


@pytest.mark.parametrize("fid,threshold", RAY_CAST_VIEWS)
def test_ray_cast_is_the_reference_ray_cast(ref, fid, threshold):
    """RayCastCPU<float, uint16_t, uint16_t> (VoxelBlockGridImpl.h:578-1120), all ten renderings, on the oracle-fused
    volume: bit-exact everywhere.  (The oracle's two clamps — voxel index res-1, range cell — cannot trigger here:
    640x480 is a multiple of the down factor, and a voxel coordinate that rounds up to `resolution` would show up as a
    mismatch.)"""
    vol = oracle_volume()
    o = vol["o"]
    E = oracle.inverse_transformation(camera_pose(fid))
    keys = np.ascontiguousarray(vol["keys"][: vol["size"]])
    rng = oracle.estimate_range(keys, PRIMESENSE_K, E, 480, 640, 8, RES, VOXEL, DMIN, DMAX)
    got = oracle.ray_cast(vol["keys"], vol["size"], o["tsdf"], o["wt"], o["col"], rng, PRIMESENSE_K, E, 480, 640,
                          RAY_CAST_ATTRS, RES, VOXEL, SCALE, DMIN, DMAX, threshold, TRUNC, 8)
    hit = got["depth"][..., 0] > 0
    assert hit.mean() > (0.5 if fid != 140 else 0.01)
    for name in RAY_CAST_ATTRS:
        ref.check(f"ray_cast_{fid}_{name}", got[name])
