"""MeshGenerator::cut_depth_maps on the device (smvsb_cut_depth_maps) against
the reference's own function: lib/mesh_generator.cc is compiled verbatim into
oracle/_ref and called on synthetic multi-view depth / normal maps. fp32 in
the reference's operation order, the three double comparisons in double: the
cut maps must be EQUAL."""
import os

import numpy as np
import pytest

from smvs_b200 import api
from oracle import ref as oref

pytestmark = pytest.mark.skipif(not oref.available(), reason="oracle/_ref not built")


def surface(x, y):
    return 5.0 + 0.3 * np.sin(1.1 * x) * np.cos(0.9 * y) + 0.05 * x


def surface_grad(x, y):
    return (0.3 * 1.1 * np.cos(1.1 * x) * np.cos(0.9 * y) + 0.05,
            -0.3 * 0.9 * np.sin(1.1 * x) * np.sin(0.9 * y))


def make_views(n, w, h, seed, normal_sign=-1.0):
    """n pinhole views of the height field z = surface(x, y): cameras near the
    plane z = 0 looking along +z with small rotations. Depth maps in MVE
    convention (distance along the ray), normal maps in world space, facing
    the cameras (normal_sign = -1; +1 gives back-facing normals, which the cut
    removes altogether); a few
    regions are pushed off the surface or removed so that every branch of the
    cut runs."""
    rng = np.random.default_rng(seed)
    flen = np.full(n, 1.1, np.float32)
    rots, transs, depths, normals = [], [], [], []
    ys, xs = np.mgrid[0:h, 0:w]
    for k in range(n):
        ang = rng.uniform(-0.06, 0.06, size=3)
        cx, cy, cz = np.cos(ang), np.sin(ang), None
        Rx = np.array([[1, 0, 0], [0, cx[0], -cy[0]], [0, cy[0], cx[0]]])
        Ry = np.array([[cx[1], 0, cy[1]], [0, 1, 0], [-cy[1], 0, cx[1]]])
        Rz = np.array([[cx[2], -cy[2], 0], [cy[2], cx[2], 0], [0, 0, 1]])
        R = (Rz @ Ry @ Rx).astype(np.float32).astype(np.float64)   # world -> cam
        c = np.array([0.6 * np.cos(2 * np.pi * k / n), 0.6 * np.sin(2 * np.pi * k / n),
                      rng.uniform(-0.1, 0.1)])
        t = (-R @ c).astype(np.float32).astype(np.float64)
        c = -R.T @ t
        ax = float(flen[k]) * max(w, h)
        dirs_cam = np.stack([(xs + 0.5 - 0.5 * w) / ax, (ys + 0.5 - 0.5 * h) / ax,
                             np.ones_like(xs, dtype=np.float64)], axis=-1)
        dirs_cam /= np.linalg.norm(dirs_cam, axis=-1, keepdims=True)
        dirs = dirs_cam @ R                       # cam -> world: R^T d
        tt = np.full((h, w), 5.0)
        for _ in range(12):
            px, py = c[0] + tt * dirs[..., 0], c[1] + tt * dirs[..., 1]
            tt = (surface(px, py) - c[2]) / dirs[..., 2]
        px, py = c[0] + tt * dirs[..., 0], c[1] + tt * dirs[..., 1]
        gx, gy = surface_grad(px, py)
        nrm = np.stack([-gx, -gy, np.ones_like(gx)], axis=-1)
        nrm /= np.linalg.norm(nrm, axis=-1, keepdims=True)
        d = tt.astype(np.float32)
        # disturbances: holes, a slab closer to the camera, a slab further away
        d[rng.random(d.shape) < 0.01] = 0.0
        y0, x0 = int(rng.integers(0, h - 40)), int(rng.integers(0, w - 60))
        d[y0:y0 + 40, x0:x0 + 60] *= np.float32(0.9)
        y0, x0 = int(rng.integers(0, h - 40)), int(rng.integers(0, w - 60))
        d[y0:y0 + 40, x0:x0 + 60] *= np.float32(1.08)
        y0, x0 = int(rng.integers(0, h - 30)), int(rng.integers(0, w - 30))
        d[y0:y0 + 30, x0:x0 + 30] = 0.0
        rots.append(R.reshape(9))
        transs.append(t)
        depths.append(d)
        normals.append((normal_sign * nrm).astype(np.float32))
    return flen, np.array(rots, np.float32), np.array(transs, np.float32), depths, normals


def test_oracle_cut_depth_maps_runs_and_cuts():
    """CPU: the compiled reference cuts the disturbed regions and keeps most of
    the consistent surface (pins the sign / convention of the synthetic maps)."""
    kept = {}
    for sign in (1.0, -1.0):
        flen, rot, trans, depths, normals = make_views(3, 160, 120, 1, sign)
        outs, inv, ctw, KR, t = oref.cut_depth_maps(flen, rot, trans, depths, normals)
        kept[sign] = np.mean([(o > 0).mean() for o in outs])
        for o, d in zip(outs, depths):
            assert np.all((o == 0) | (o == d))          # a cut only removes
    # the cut leaves a surface point in the view that sees it best: ~1/n of the
    # overlap survives per view; back-facing normals (sign +1) leave nothing
    assert kept[-1.0] > 0.3 and kept[1.0] == 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("n,w,h", [(3, 160, 120), (5, 320, 240), (4, 333, 207),
                                   (7, 1920, 1080)])
def test_cut_depth_maps_equal_to_reference(n, w, h):
    """The last case is BASELINE.json's view size: 7 views at 1920x1080."""
    import json
    import time
    flen, rot, trans, depths, normals = make_views(n, w, h, n)
    t0 = time.perf_counter()
    outs, inv, ctw, KR, t = oref.cut_depth_maps(flen, rot, trans, depths, normals)
    t_cpu = time.perf_counter() - t0
    api.cut_depth_maps(depths, normals, inv, ctw, KR, t)          # warm-up
    t0 = time.perf_counter()
    got = api.cut_depth_maps(depths, normals, inv, ctw, KR, t)
    t_gpu = time.perf_counter() - t0
    print(json.dumps({"cut_depth_maps": f"{n} views {w}x{h}",
                      "reference_s_4_threads": t_cpu, "abi_call_s": t_gpu}))
    kept, cut = 0, 0
    for g, o, d in zip(got, outs, depths):
        assert np.array_equal(g, o)
        kept += int((o > 0).sum())
        cut += int(((o == 0) & (d > 0)).sum())
    assert kept > 0.15 * n * w * h and cut > 0.03 * n * w * h


@pytest.mark.gpu
@pytest.mark.skipif(not os.path.exists(oref.INTEGRATION_LIB_PATH),
                    reason="oracle/_ref/integration not built")
def test_cut_depth_maps_drop_in_member():
    """MeshGenerator::cut_depth_maps of the drop-in build (integration/
    b200_mesh_generator.cc: the reference's MeshGenerator object, cameras and
    ViewProjections, the cut on the GPU) against the pure-CPU build."""
    flen, rot, trans, depths, normals = make_views(4, 320, 240, 11)
    cpu = oref.cut_depth_maps(flen, rot, trans, depths, normals)[0]
    before = api.lib().smvsb_global_launch_count()
    gpu = oref.cut_depth_maps(flen, rot, trans, depths, normals,
                              lib_path=oref.INTEGRATION_LIB_PATH)[0]
    assert api.lib().smvsb_global_launch_count() > before
    for g, c in zip(gpu, cpu):
        assert np.array_equal(g, c)
