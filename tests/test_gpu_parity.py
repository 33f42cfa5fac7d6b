"""Parity of the CUDA path (through the C ABI of include/smvs_b200.h) against
(1) the committed golden fixtures and (2) the compiled-verbatim reference
run live on the same seeded inputs.

Tolerances. The Gauss-Newton path is fp64; the cancellation-prone per-sample
quantities are evaluated bitwise like the reference (gn_math.cuh: xd), the
accumulation has a different (but fixed) summation order, so values agree to
~1e-14 relative; the tests ask for 1e-11 on g / H, 1e-7..1e-8 on P and the CG
solution (conditioning) and for EQUAL iteration counts and active sets. Depth maps (float32 outputs) must agree to 1e-6 relative,
far inside the 1e-4 of BASELINE.json. SGM is integer work: bit-exact."""
import os

import numpy as np
import pytest

from smvs_b200 import api, synth
from oracle import ref as oref

from util_scene import Pair, RefOutputs, rel_err

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TOL = 1e-11


def load(name):
    return np.load(os.path.join(GOLD, name), allow_pickle=False)


def ctx_from_golden(G):
    ctx = api.Context(0)
    n = int(G["n_sub"])
    sh = G["shading"] if "shading" in G else None
    shg = G["shading_grad"] if "shading_grad" in G else None
    ctx.set_views(G["main_grad"], [G[f"sub_grad{k}"] for k in range(n)],
                  [G[f"sub_hess{k}"] for k in range(n)], G["Mi"], G["ti"],
                  float(G["flen"]), float(G["inv_flen"]), sh, shg)
    ctx.set_surface(int(G["scale"]), int(G["npx"]), int(G["npy"]), int(G["start_x"]),
                    int(G["start_y"]), G["nodes"], G["node_valid"], G["patch_valid"],
                    G["vis_off"], G["vis_ids"])
    return ctx


def _diag_positions(sysd):
    """Indices into Hvals of the diagonal blocks, in column order."""
    outer, inner = sysd["Houter"], sysd["Hinner"]
    out = []
    for col in range(len(outer) - 1):
        for k in range(int(outer[col]), int(outer[col + 1])):
            if int(inner[k]) == 4 * col:
                out.append(k)
    return np.array(out, dtype=np.int64)


def assert_system_equal(gs, rs):
    assert np.array_equal(gs["Houter"], rs["Houter"])
    assert np.array_equal(gs["Hinner"], rs["Hinner"])
    assert np.array_equal(gs["Pouter"], rs["Pouter"])
    assert np.array_equal(gs["Pinner"], rs["Pinner"])
    assert rel_err(gs["g"], rs["g"]) < TOL
    assert rel_err(gs["Hvals"], rs["Hvals"]) < TOL
    # P = inverse of the diagonal block. Where that block is numerically
    # singular (scale 0: one sample per patch) the LDL^T "inverse" is rounding
    # noise times 1e16 in the reference as well; compare the blocks whose
    # condition estimate |D| * |D^-1| is sane.
    diag = rs["Hvals"][np.isin(np.arange(len(rs["Hinner"])), _diag_positions(rs))]
    cond = np.abs(diag).max(axis=1) * np.abs(rs["Pvals"]).max(axis=1)
    well = cond < 1e8
    assert well.mean() > 0.5 or len(well) == 0 or rs["Houter"].size < 8000
    if well.any():
        assert rel_err(gs["Pvals"][well], rs["Pvals"][well]) < 1e-7


@pytest.mark.parametrize("fixture", ["gn_s2.npz", "gn_s4.npz"])
def test_golden_construct_cg(fixture):
    G = load(fixture)
    with ctx_from_golden(G) as ctx:
        for tag in G["variants"]:
            light = G["light"] if tag in ("lit", "litR") else None
            ctx.gn_construct(G[f"{tag}_active"], light, float(G["regularization"]),
                             float(G[f"{tag}_lreg"]))
            gs = ctx.debug_get_system()
            rs = {k: G[f"{tag}_{k}"] for k in
                  ("g", "Hvals", "Houter", "Hinner", "Pvals", "Pouter", "Pinner")}
            assert_system_equal(gs, rs)
            it, info = ctx.cg_solve()
            assert it == int(G[f"{tag}_cg_iters"]) and info == int(G[f"{tag}_cg_info"])
            assert rel_err(ctx.get_delta(), G[f"{tag}_x"]) < 1e-8


@pytest.mark.parametrize("fixture", ["gn_s2.npz", "gn_s4.npz"])
def test_golden_update_and_loop(fixture):
    G = load(fixture)
    with ctx_from_golden(G) as ctx:
        ctx.gn_construct(G["full_active"], None, float(G["regularization"]), 0.0)
        ctx.cg_solve()
        act, n_act, shift = ctx.update_nodes()
        assert np.array_equal(act, G["upd_active"])
        assert n_act == int(G["upd_n_active"])
        assert abs(shift - float(G["upd_mean_shift"])) < 1e-9 * max(1.0, abs(shift))
        assert rel_err(ctx.get_nodes(), G["upd_nodes"]) < TOL

        ctx.set_nodes(G["nodes"])
        light = G["light"] if "light" in G else None
        st = ctx.newton_loop(light, float(G["regularization"]), 0.0)
        assert st["newton_steps"] == int(G["loop_newton_steps"])
        assert st["cg_iterations"] == int(G["loop_cg_iterations"])
        assert st["pixel_iterations"] == float(G["loop_pixel_iterations"])
        assert st["n_active"] == int(G["loop_n_active"])
        assert rel_err(ctx.get_nodes(), G["loop_nodes"]) < 1e-8
        d, dr = ctx.get_depth(), G["loop_depth"]
        assert np.array_equal(d > 0, dr > 0)
        assert rel_err(d, dr) < 1e-6
        assert np.max(np.abs(ctx.get_normals() - G["loop_normals"])) < 1e-6


def test_golden_sgm_bit_exact():
    G = load("sgm.npz")
    r = api.sgm(G["main"], G["neigh"], G["M"], G["t"], float(G["min_depth"]),
                float(G["max_depth"]), int(G["D"]), volumes=True)
    assert np.array_equal(r["cost"], G["cost"].astype(np.uint16))
    assert np.array_equal(r["sgm"], G["sgm"])
    assert np.array_equal(r["depth"], G["depth"])


@pytest.mark.parametrize("w,h", [(333, 207), (352, 207)])
def test_device_set_scale_bitwise(w, h):
    """smvsb_set_views_u8 (StereoView::set_scale on the device) against the
    numpy mirror, which tests/test_cpu_host.py pins bitwise to the reference.
    Row pitches that are a multiple of 16 bytes take the TMA-staged fused
    kernel, the others the three separate kernels: both must give the same
    bits, at blur radii from 2 (scale 2) to 12 (scale 5)."""
    from smvs_b200 import stereo_view, workload
    sc = synth.make_scene(w, h, 2, seed_index=4, shading=True)
    for scale in (2, 3, 5):
        wl = workload.build_workload(w, h, 2, scale=scale, scene=sc, shading=True)
        with api.Context(0) as ctx:
            wl.push_views_u8(ctx)
            g, _ = ctx.debug_get_view(0)
            assert np.array_equal(g, wl.main_grad)
            for k in range(2):
                g, hs = ctx.debug_get_view(k + 1)
                assert np.array_equal(g, wl.sub_grads[k])
                assert np.array_equal(hs, wl.sub_hess[k])
            # the Gauss-Newton system built from device-made inputs is the one
            # built from host-made inputs, bit for bit (shading path included)
            wl.push_surface(ctx)
            light = np.linspace(1.0, -0.2, 16)
            ctx.gn_construct(None, light, 0.01, 0.0)
            a = ctx.debug_get_system()
            wl.push_views(ctx)
            wl.push_surface(ctx)
            ctx.gn_construct(None, light, 0.01, 0.0)
            b = ctx.debug_get_system()
            assert np.array_equal(a["g"], b["g"]) and np.array_equal(a["Hvals"], b["Hvals"])


@pytest.mark.gpu
def test_view_set_scale_colour_bitwise():
    """smvsb_view_set_scale_c on three-channel views: channel-wise Gaussian
    blur, luminance of the blurred image, gradient / Hessian stencil
    (lib/stereo_view.cc:24-62) -- scaleimage, gradients and Hessian bitwise
    the compiled reference's."""
    from smvs_b200 import stereo_view
    from util_scene import colour_scene
    ref = RefOutputs("view_set_scale_colour")
    sc = colour_scene(333, 207, 2, 71)
    R = oref.RefScene(sc) if ref.live else None
    try:
        with api.Context(0) as ctx:
            for scale in (0, 2, 3, 5):
                if R:
                    R.set_scale(scale)
                for v in range(3):
                    img = stereo_view.byte_to_float(sc.images[v])
                    assert img.shape == (207, 333, 3)
                    k = f"s{scale}v{v}"
                    ref.assert_equal(k + "/image", img, lambda: R.image(v))
                    blur, grad, hess = ctx.view_set_scale(img, scale)
                    ref.assert_equal(k + "/blur", blur, lambda: R.scaleimage(v))
                    ref.assert_equal(k + "/grad", grad, lambda: R.gradients(v))
                    ref.assert_equal(k + "/hess", hess, lambda: R.hessian(v))
    finally:
        if R:
            R.close()


def test_view_set_scale_bitwise():
    """smvsb_view_set_scale (one StereoView::set_scale, host image in, host
    images out -- what the drop-in member calls) against the numpy mirror."""
    from smvs_b200 import stereo_view
    for w in (333, 336):          # 336 * 4 bytes: the TMA-staged fused kernel
        sc = synth.make_scene(w, 207, 1, seed_index=5)
        img = sc.images[1]
        with api.Context(0) as ctx:
            for scale in (0, 2, 4, 6):
                f = stereo_view.byte_to_float(img)
                blur, grad, hess = ctx.view_set_scale(f, scale)
                rb, rg, rh = stereo_view.set_scale(img, scale)
                assert np.array_equal(blur, rb)
                assert np.array_equal(grad, rg) and np.array_equal(hess, rh)


def test_bilateral_filter_bit_exact():
    """smvsb_bilateral_filter against DepthOptimizer::depthmap_bilateral_filter
    (joint bilateral filter of the SGM init): fp32 with expf in the loop --
    bit-identical, full-resolution and half-resolution depth, with holes."""
    from smvs_b200 import stereo_view
    ref = RefOutputs("bilateral_filter")
    sc = synth.make_scene(333, 207, 1, seed_index=6)
    R = oref.RefScene(sc) if ref.live else None
    guide = stereo_view.byte_to_float(sc.images[0])
    ref.assert_equal("guide", guide, lambda: R.image(0))
    d = sc.init_depth.astype(np.float32).copy()
    d[::7, ::5] = 0.0
    d[40:80, 100:160] = 0.0
    with api.Context(0) as ctx:
        for k, dm in enumerate((d, d[::2, ::2].copy())):
            out = ctx.bilateral_filter(guide, dm)
            ref.assert_equal(f"depth{k}", out, lambda: R.bilateral_filter(dm))
            assert (out > 0).mean() > 0.8
    if R:
        R.close()


# ---------------------------------------------------------------------------
# live reference, larger / odd shapes
# ---------------------------------------------------------------------------

needs_ref = pytest.mark.skipif(not oref.available(), reason="oracle/_ref not built")


@needs_ref
@pytest.mark.parametrize("w,h,n_sub,scale", [(640, 480, 2, 2), (640, 480, 3, 3),
                                             (417, 311, 2, 4), (640, 480, 6, 5),
                                             (96, 72, 2, 0), (160, 120, 2, 1),
                                             (640, 480, 2, 6)])
def test_live_construct_parity(w, h, n_sub, scale):
    P = Pair(w, h, n_sub, scale)
    try:
        rng = np.random.default_rng(scale)
        full = P.node_valid.copy()
        part = (full & (rng.random(full.shape) < 0.25)).astype(np.uint8)
        none = np.zeros_like(full)
        for act, reg in ((full, 0.01), (part, 0.01), (full, 0.0)):
            P.R.gn_construct(act, None, reg, 0.0)
            P.ctx.gn_construct(act, None, reg, 0.0)
            assert_system_equal(P.ctx.debug_get_system(), P.R.get_system())
            x = rng.standard_normal(P.ctx.n_nodes * 4)
            assert rel_err(P.ctx.debug_spmv(x), P.R.hessian_multiply(x)) < TOL
        # empty active set: empty system, lib/gauss_newton_step.cc:73-79
        P.ctx.gn_construct(none, None, 0.01, 0.0)
        gs = P.ctx.debug_get_system()
        assert len(gs["Hvals"]) == 0 and not gs["g"].any()
    finally:
        P.close()


@needs_ref
def test_live_ragged_surface_and_neighbour_sizes():
    """Holes in the surface, patches with 0..n visible neighbours."""
    P = Pair(400, 300, 3, 2, seed_index=5, gpu=True)
    try:
        rng = np.random.default_rng(3)
        pv = P.patch_valid.copy()
        pv[rng.random(pv.shape) < 0.2] = 0
        npx, npy = P.info["npx"], P.info["npy"]
        nv = np.zeros_like(P.node_valid)
        pv2 = pv.reshape(npy, npx)
        nv2 = nv.reshape(npy + 1, npx + 1)
        for dy in (0, 1):
            for dx in (0, 1):
                nv2[dy:dy + npy, dx:dx + npx] |= pv2
        P.node_valid, P.patch_valid = nv, pv
        P.R.surface_set(P.nodes, nv, pv)
        # thin the visibility lists at random
        off, ids = [0], []
        for p in range(npx * npy):
            lst = [i for i in P.vis_ids[P.vis_off[p]:P.vis_off[p + 1]] if rng.random() < 0.7]
            if pv[p] and not lst:
                lst = [int(rng.integers(0, 3))]
            ids += lst
            off.append(len(ids))
        P.vis_off, P.vis_ids = np.array(off, np.uint32), np.array(ids, np.uint8)
        P.R.set_visibility(P.vis_off, P.vis_ids)
        P.push_surface()
        P.R.gn_construct(nv, None, 0.01, 0.0)
        P.ctx.gn_construct(nv, None, 0.01, 0.0)
        assert_system_equal(P.ctx.debug_get_system(), P.R.get_system())
        xr, itr, _ = P.R.cg_solve()
        itg, _ = P.ctx.cg_solve()
        assert itg == itr and rel_err(P.ctx.get_delta(), xr) < 1e-8
        ar, nr, _ = P.R.update_nodes(xr, nv)
        ag, ng, _ = P.ctx.update_nodes()
        assert ng == nr and np.array_equal(ag, ar)
    finally:
        P.close()


@needs_ref
def test_live_shading_newton_loop():
    P = Pair(640, 480, 3, 2, shading=True)
    try:
        lr, lg = P.R.fit_lighting(), P.ctx.fit_lighting()
        # 16x16 pseudo inverse of an ill-conditioned normal matrix
        assert rel_err(lg, lr) < 1e-5
        for lreg in (0.0, 5.0):
            P.R.gn_construct(P.node_valid, lr, 0.01, lreg)
            P.ctx.gn_construct(P.node_valid, lr, 0.01, lreg)
            assert_system_equal(P.ctx.debug_get_system(), P.R.get_system())
        sr = P.R.newton_loop(lr, 0.01, 0.0)
        sg = P.ctx.newton_loop(lr, 0.01, 0.0)
        for k in ("newton_steps", "cg_iterations", "n_active", "pixel_iterations"):
            assert sg[k] == sr[k], k
        d, dr = P.ctx.get_depth(), P.R.surface_depth()
        assert np.array_equal(d > 0, dr > 0) and rel_err(d, dr) < 1e-6
    finally:
        P.close()


@needs_ref
@pytest.mark.parametrize("w,h,scale", [(160, 120, 1), (640, 480, 6)])
def test_live_newton_loop_extreme_scales(w, h, scale):
    """1, 4 and 256 samples per patch (-o0, -o1, and the no-SGM start scale)."""
    P = Pair(w, h, 2, scale)
    try:
        sr = P.R.newton_loop(None, 0.01, 0.0)
        sg = P.ctx.newton_loop(None, 0.01, 0.0)
        for k in ("newton_steps", "cg_iterations", "n_active", "pixel_iterations"):
            assert sg[k] == sr[k], k
        d, dr = P.ctx.get_depth(), P.R.surface_depth()
        assert np.array_equal(d > 0, dr > 0) and rel_err(d, dr) < 1e-6
    finally:
        P.close()


@needs_ref
def test_live_full_opt_mean_shift():
    P = Pair(320, 240, 2, 3)
    try:
        P.R.gn_construct(P.node_valid, None, 0.01, 0.0)
        P.ctx.gn_construct(P.node_valid, None, 0.01, 0.0)
        xr, _, _ = P.R.cg_solve()
        P.ctx.cg_solve()
        ar, nr, mr = P.R.update_nodes(xr, P.node_valid, full_opt=True)
        ag, ng, mg = P.ctx.update_nodes(full_opt=True)
        assert abs(mg - mr) < 1e-9 * max(abs(mr), 1e-12)
        assert np.array_equal(ag, ar)     # unchanged in full_opt mode
    finally:
        P.close()


def _sgm_against_reference(ref, sc, dmin, dmax, D):
    w, h = sc.width, sc.height
    R = oref.RefScene(sc) if ref.live else None
    r = R.sgm_run(0, 1, 0, D, dmin, dmax, volumes=True) if R else None
    M = ref.array("M", lambda: R.reprojection(0, 1, w, h, w, h)[0])
    t = ref.array("t", lambda: R.reprojection(0, 1, w, h, w, h)[1])
    g = api.sgm(sc.images[0], sc.images[1], M, t, dmin, dmax, D, volumes=True)
    for k in ("cost", "sgm", "depth"):
        ref.assert_equal(k, g[k], lambda: r[k])
    if R:
        R.close()


@pytest.mark.parametrize("w,h,D", [(333, 207, 64), (640, 480, 128), (200, 150, 32)])
def test_live_sgm_bit_exact(w, h, D):
    sc = synth.make_scene(w, h, 1, seed_index=9)
    dmin, dmax = float(sc.true_depth.min() * 0.7), float(sc.true_depth.max() * 1.3)
    _sgm_against_reference(RefOutputs(f"sgm_{w}x{h}x{D}"), sc, dmin, dmax, D)


def test_live_sgm_low_texture_and_behind_camera():
    """Zero / dark pixels (census skipped, luminance < 25 rejected) and a depth
    range that puts planes behind the neighbour camera."""
    sc = synth.make_scene(256, 192, 1, seed_index=10)
    sc.images[0][40:80, 50:120] = 0
    sc.images[0][100:140, 30:90] = 12
    sc.images[1][60:100, 100:200] = 0
    _sgm_against_reference(RefOutputs("sgm_low_texture"), sc, 0.05, 40.0, 64)


# ---------------------------------------------------------------------------
# BASELINE.json sizes: size-independent properties + one live comparison
# ---------------------------------------------------------------------------

def test_full_size_properties():
    """1920x1080, 6 neighbours, scale 2: H symmetric, SpMV linear, CG
    solution satisfies the reference's stopping rule, deterministic rerun."""
    from bench import build_workload
    wl = build_workload(1920, 1080, 6, scale=2, shading=False)
    with api.Context(0) as ctx:
        wl.push(ctx)
        ctx.gn_construct(None, None, 0.01, 0.0)
        rng = np.random.default_rng(0)
        n = ctx.n_nodes * 4
        x, y = rng.standard_normal(n), rng.standard_normal(n)
        Hx, Hy = ctx.debug_spmv(x), ctx.debug_spmv(y)
        assert abs(np.dot(y, Hx) - np.dot(x, Hy)) < 1e-9 * abs(np.dot(y, Hx))
        assert rel_err(ctx.debug_spmv(2.0 * x - 3.0 * y), 2.0 * Hx - 3.0 * Hy) < 1e-12
        assert np.dot(x, Hx) > 0.0                       # J^T J is PSD
        it, info = ctx.cg_solve()
        d1 = ctx.get_delta()
        g = ctx.debug_get_system()["g"]
        res = ctx.debug_spmv(d1) + g
        assert np.linalg.norm(res) < np.linalg.norm(g)
        it2, _ = ctx.cg_solve()
        assert it2 == it and np.array_equal(ctx.get_delta(), d1)   # deterministic


# ---------------------------------------------------------------------------
# error behaviour of the ABI (codes instead of the reference's exceptions)
# ---------------------------------------------------------------------------

def test_error_paths():
    G = load("gn_s2.npz")
    n = int(G["n_sub"])
    views = dict(main_grad=G["main_grad"], sub_grads=[G[f"sub_grad{k}"] for k in range(n)],
                 sub_hess=[G[f"sub_hess{k}"] for k in range(n)], Mi=G["Mi"], ti=G["ti"],
                 flen_px=float(G["flen"]), inv_flen=float(G["inv_flen"]))
    surf = [int(G["scale"]), int(G["npx"]), int(G["npy"]), int(G["start_x"]),
            int(G["start_y"]), G["nodes"], G["node_valid"], G["patch_valid"],
            G["vis_off"], G["vis_ids"]]
    with api.Context(0) as ctx:
        with pytest.raises(api.SmvsbError) as e:       # call order
            ctx.set_surface(*surf)
        assert e.value.code == -4
        ctx.set_views(**views)
        with pytest.raises(api.SmvsbError) as e:       # no system yet
            ctx.n_nodes = 10
            ctx.cg_solve()
        assert e.value.code == -4
        bad = list(surf)
        bad[0] = 7                                     # unsupported scale
        with pytest.raises(api.SmvsbError) as e:
            ctx.set_surface(*bad)
        assert e.value.code == -1
        bad = list(surf)
        bad[1] = surf[1] + 50                          # grid larger than the image
        bad[5] = np.zeros(((bad[1] + 1) * (surf[2] + 1), 4))
        bad[6] = np.zeros((bad[1] + 1) * (surf[2] + 1), np.uint8)
        bad[7] = np.zeros(bad[1] * surf[2], np.uint8)
        bad[8] = np.zeros(bad[1] * surf[2] + 1, np.uint32)
        with pytest.raises(api.SmvsbError) as e:
            ctx.set_surface(*bad)
        assert e.value.code == -1
        bad = list(surf)
        bad[9] = np.full_like(surf[9], 9)              # neighbour id out of range
        with pytest.raises(api.SmvsbError) as e:
            ctx.set_surface(*bad)
        assert e.value.code == -1
        if surf[9].size >= 2 and surf[8][1] >= 2:
            bad = list(surf)
            bad[9] = surf[9].copy()
            bad[9][1] = bad[9][0]                      # a neighbour twice in one list
            with pytest.raises(api.SmvsbError) as e:
                ctx.set_surface(*bad)
            assert e.value.code == -1
            assert b"duplicate" in api.lib().smvsb_last_error(ctx._h)
        bad = list(surf)
        bad[8] = surf[8].copy()
        bad[8][1], bad[8][2] = surf[8][2] + 1, surf[8][1]   # offsets not monotone
        with pytest.raises(api.SmvsbError) as e:
            ctx.set_surface(*bad)
        assert e.value.code == -1
        # a failed call leaves the context without a surface
        with pytest.raises(api.SmvsbError):
            ctx.gn_construct(None, None, 0.01, 0.0)
        ctx.set_surface(*surf)
        with pytest.raises(api.SmvsbError) as e:       # lighting without shading image
            ctx.gn_construct(None, np.ones(16), 0.01, 0.0)
        assert e.value.code == -4
        ctx.gn_construct(None, None, 0.01, 0.0)        # still usable afterwards
        assert ctx.cg_solve()[0] > 0
    z = np.zeros((64, 64), np.uint8)
    eye, t0 = np.eye(3, dtype=np.float32).ravel(), np.zeros(3, np.float32)
    for kwargs in (dict(num_steps=48), dict(penalty1=100, penalty2=50),
                   dict(penalty2=300)):
        with pytest.raises(api.SmvsbError) as e:
            api.sgm(z, z, eye, t0, 1.0, 2.0, **kwargs)
        assert e.value.code == -1
    with pytest.raises(api.SmvsbError):                # image smaller than the census
        api.sgm(z[:6, :8], z, eye, t0, 1.0, 2.0)


def test_nan_break_and_zero_gradient():
    """Constant images: zero photometric gradient everywhere. The loop must
    leave through the reference's NaN rule or converge, never hang."""
    G = load("gn_s4.npz")
    n = int(G["n_sub"])
    with api.Context(0) as ctx:
        zero2 = np.zeros_like(G["main_grad"])
        ctx.set_views(zero2, [np.zeros_like(G[f"sub_grad{k}"]) for k in range(n)],
                      [np.zeros_like(G[f"sub_hess{k}"]) for k in range(n)], G["Mi"],
                      G["ti"], float(G["flen"]), float(G["inv_flen"]))
        ctx.set_surface(int(G["scale"]), int(G["npx"]), int(G["npy"]), int(G["start_x"]),
                        int(G["start_y"]), G["nodes"], G["node_valid"], G["patch_valid"],
                        G["vis_off"], G["vis_ids"])
        st = ctx.newton_loop(None, 0.0, 0.0, max_steps=5)   # no regulariser: g = 0, H = 0
        assert st["nan"] and st["newton_steps"] == 1
        assert np.array_equal(ctx.get_nodes(), G["nodes"])  # surface untouched


@needs_ref
@pytest.mark.parametrize("shading", [False, True])
def test_full_size_live_parity(shading):
    """BASELINE.json configs[1] / configs[2] at their real size (1 ref + 6
    neighbours, 1920x1080, scale 2): one Gauss-Newton construct + PCG solve +
    update against the compiled reference on the bench workload's own
    arrays."""
    from bench import _ref_scene_for
    from smvs_b200.workload import build_workload
    wl = build_workload(1920, 1080, 6, scale=2, shading=shading, seed_index=3)
    R = _ref_scene_for(wl)
    with api.Context(0) as ctx:
        wl.push_views_u8(ctx)          # device set_scale, bit-identical inputs
        wl.push_surface(ctx)
        light = None
        if shading:
            light, lg = R.fit_lighting(), ctx.fit_lighting()
            assert rel_err(lg, light) < 1e-5
        act = wl.node_valid
        R.gn_construct(act, light, 0.01, 0.0)
        ctx.gn_construct(act, light, 0.01, 0.0)
        rs, gs = R.get_system(), ctx.debug_get_system()
        assert np.array_equal(gs["Hinner"], rs["Hinner"])
        assert rel_err(gs["g"], rs["g"]) < TOL
        assert rel_err(gs["Hvals"], rs["Hvals"]) < TOL
        xr, itr, infr = R.cg_solve()
        itg, infg = ctx.cg_solve()
        assert (itg, infg) == (itr, infr)
        # the first solve at 2 MP runs into max_iterations (199 updates of an
        # unconverged Krylov process): rounding differences of 1e-15 in H are
        # amplified to ~1e-5 in x by the loss of orthogonality, in any
        # implementation. The update step is therefore compared on the
        # reference's own x.
        assert rel_err(ctx.get_delta(), xr) < 1e-3
        ctx.set_delta(xr)
        ar, nr, _ = R.update_nodes(xr, act)
        ag, ng, _ = ctx.update_nodes()
        assert ng == nr and np.array_equal(ag, ar)
        valid = wl.node_valid.astype(bool)      # the reference reports 0 for null nodes
        assert np.array_equal(ctx.get_nodes()[valid], R.surface_get()[0][valid])
    R.close()


# ---------------------------------------------------------------------------
# several views per launch (smvsb_newton_loop_batch)
# ---------------------------------------------------------------------------

def test_batch_is_bitwise_the_single_view_loop():
    """Views of different sizes, with and without lighting, advanced in
    lock-step with one PCG launch per step: every view's nodes, step and
    iteration counts are EXACTLY those of its own smvsb_newton_loop (the
    reference runs the views independently, app/smvsrecon.cc:658-733)."""
    from smvs_b200 import workload
    specs = [(640, 480, 3, 2, False, 11), (400, 300, 2, 2, True, 12),
             (640, 480, 2, 3, False, 13), (333, 207, 2, 2, True, 14),
             (96, 72, 2, 2, False, 15)]
    wls = [workload.build_workload(w, h, n, scale=s, shading=sh, seed_index=seed)
           for (w, h, n, s, sh, seed) in specs]
    ctxs = [api.Context(0) for _ in wls]
    try:
        lights, single, nodes_single = [], [], []
        for wl, ctx in zip(wls, ctxs):
            wl.push_views_u8(ctx)
            wl.push_surface(ctx)
            lights.append(ctx.fit_lighting() if wl.shading is not None else None)
        for wl, ctx, light in zip(wls, ctxs, lights):
            single.append(ctx.newton_loop(light, 0.01, 0.0))
            nodes_single.append(ctx.get_nodes())
            ctx.set_nodes(wl.nodes)
        before = sum(c.launches for c in ctxs)
        batch = api.newton_loop_batch(ctxs, lights, 0.01, 0.0)
        assert sum(c.launches for c in ctxs) > before
        for k, (ctx, s, b) in enumerate(zip(ctxs, single, batch)):
            for key in ("newton_steps", "cg_iterations", "n_active", "pixel_iterations",
                        "nan", "cg_block_iterations", "cg_row_iterations"):
                assert b[key] == s[key], (k, key, b[key], s[key])
            assert np.array_equal(ctx.get_nodes(), nodes_single[k]), k
        # a batch of one is the plain loop
        ctxs[0].set_nodes(wls[0].nodes)
        one = api.newton_loop_batch(ctxs[:1], None, 0.01, 0.0)[0]
        assert one["cg_iterations"] == single[0]["cg_iterations"]
        assert np.array_equal(ctxs[0].get_nodes(), nodes_single[0])
        # error paths: the same context twice, too many contexts
        with pytest.raises(api.SmvsbError) as e:
            api.newton_loop_batch([ctxs[0], ctxs[0]], None, 0.01, 0.0)
        assert e.value.code == -1
        with pytest.raises(api.SmvsbError) as e:
            api.newton_loop_batch([ctxs[k % 5] for k in range(9)], None, 0.01, 0.0)
        assert e.value.code == -1
    finally:
        for c in ctxs:
            c.close()


def test_sgm_reconstruct_and_merge_bit_exact():
    """smvsb_sgm_reconstruct: run_sgm in both directions, the consistency check
    (lib/sgm_stereo.cc:64-91) and the two-neighbour merge
    (app/smvsrecon.cc:362-377) on the device, against SGMStereo::reconstruct of
    the compiled reference: the depth image that leaves the GPU is bit-exact."""
    w, h = 352, 264
    sc = synth.make_scene(w, h, 2, seed_index=23)
    dmin, dmax = float(sc.true_depth.min() * 0.7), float(sc.true_depth.max() * 1.3)
    ref = RefOutputs("sgm_reconstruct_merge")
    R = oref.RefScene(sc) if ref.live else None
    refd = [R.sgm_reconstruct(0, k, 0, 64, dmin, dmax) for k in (1, 2)] if R else None
    out, single, prev = [], [], None
    for k in (1, 2):
        M_mn = ref.array(f"M{k}", lambda: R.reprojection(0, k, w, h, w, h)[0])
        t_mn = ref.array(f"t{k}", lambda: R.reprojection(0, k, w, h, w, h)[1])
        M_nm = ref.array(f"M{k}_back", lambda: R.reprojection(k, 0, w, h, w, h)[0])
        t_nm = ref.array(f"t{k}_back", lambda: R.reprojection(k, 0, w, h, w, h)[1])
        single.append(api.sgm_reconstruct(sc.images[0], sc.images[k], M_mn, t_mn, M_nm, t_nm,
                                          (dmin, dmax), (dmin, dmax), 64)["depth"])
        ref.assert_equal(f"depth{k}", single[-1], lambda: refd[k - 1])
        assert 0.2 < (single[-1] > 0).mean() < 1.0      # the check rejects something
        prev = api.sgm_reconstruct(sc.images[0], sc.images[k], M_mn, t_mn, M_nm, t_nm,
                                   (dmin, dmax), (dmin, dmax), 64, merge_with=prev)["depth"]
        out.append(prev)
    if R:
        R.close()
    # app/smvsrecon.cc:362-377 on the two single-neighbour results, each equal
    # to the reference's
    d1, d2 = single[0].copy(), single[1]
    both = (d1 != 0) & (d2 != 0)
    only2 = (d1 == 0) & (d2 != 0)
    d1[both] = (d1[both] + d2[both]) * np.float32(0.5)
    d1[only2] = d2[only2]
    assert np.array_equal(out[0], single[0])
    assert np.array_equal(out[1], d1)
