"""CPU-side tests: the C ABI library loads and exports what the header
declares, fails loudly without a GPU, and the host-side mirrors (set_scale,
workload builder, sharding) behave like the reference."""
import ctypes as C
import os
import re
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

from smvs_b200 import api, sharding, stereo_view, synth, workload
from oracle import ref as oref


def _has_gpu():
    import torch
    return torch.cuda.is_available()


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "smvs_b200.h")).read()
    declared = set(re.findall(r"\b(smvsb_[a-z_0-9]+)\s*\(", hdr))
    declared -= {"smvsb_ctx", "smvsb_status"}
    assert declared == set(api.EXPORTS)
    L = api.lib()
    for name in sorted(declared):
        assert hasattr(L, name), name
    assert b"sm_100a" in L.smvsb_version()
    # the documents quote the number of entry points
    for doc in ("README.md", "DESIGN.md"):
        text = open(os.path.join(ROOT, doc)).read()
        assert f"{len(declared)} entry points" in text, doc


@pytest.mark.skipif(_has_gpu(), reason="checks the no-GPU failure path")
@pytest.mark.skipif(not os.path.exists(oref.INTEGRATION_LIB_PATH),
                    reason="oracle/_ref/integration not built")
def test_drop_in_build_resolves_every_symbol():
    """oracle/_ref/integration/libsmvs_ref_b200.so (reference objects + drop-in
    members + libsmvs_b200.so) loads with immediate binding: no reference member
    is left without a body, and each drop-in member is the strong definition."""
    C.CDLL(oref.INTEGRATION_LIB_PATH, mode=os.RTLD_NOW)
    import subprocess
    out = subprocess.run(["nm", "-DC", "--defined-only", oref.INTEGRATION_LIB_PATH],
                         capture_output=True, text=True).stdout
    for member in ("smvs::DepthOptimizer::optimize()",
                   "smvs::DepthOptimizer::run_newton_iterations(int)",
                   "smvs::DepthOptimizer::create_subview_surfaces()",
                   "smvs::DepthOptimizer::cut_boundaries()",
                   "smvs::StereoView::set_scale(int, bool)",
                   "smvs::SGMStereo::run_sgm(float, float)",
                   "smvs::SGMStereo::reconstruct(",
                   "smvs::MeshGenerator::cut_depth_maps("):
        lines = [ln for ln in out.splitlines() if member in ln]
        assert lines and all(" T " in ln for ln in lines), (member, lines)


def test_no_cpu_fallback():
    h = C.c_void_p()
    rc = api.lib().smvsb_create(0, C.byref(h))
    assert rc == -2 and not h
    assert b"no CPU fallback" in api.lib().smvsb_last_error(None)
    with pytest.raises(api.SmvsbError):
        api.Context(0)
    with pytest.raises(api.SmvsbError):
        z = np.zeros((64, 64), np.uint8)
        api.sgm(z, z, np.eye(3).ravel(), np.zeros(3), 1.0, 2.0, 64)


def test_null_context_is_rejected():
    L = api.lib()
    assert L.smvsb_cg_solve(None, 10, C.c_double(0), C.c_double(0), None, None) == -1
    assert L.smvsb_get_nodes(None, None) == -1


def test_synth_is_seeded():
    a = synth.make_scene(96, 64, 2, seed_index=3)
    b = synth.make_scene(96, 64, 2, seed_index=3)
    c = synth.make_scene(96, 64, 2, seed_index=4)
    assert all(np.array_equal(x, y) for x, y in zip(a.images, b.images))
    assert not np.array_equal(a.images[0], c.images[0])


def test_set_scale_mirror_matches_reference_bitwise():
    from util_scene import RefOutputs
    ref = RefOutputs("set_scale_mirror")
    sc = synth.make_scene(160, 120, 1, seed_index=2, shading=True)
    R = oref.RefScene(sc, init_linear=True) if ref.live else None
    for scale in (2, 4):
        if R:
            R.set_scale(scale)
        for v in (0, 1):
            b, g, h = stereo_view.set_scale(sc.images[v], scale)
            k = f"s{scale}v{v}"
            ref.assert_equal(k + "/blur", b, lambda: R.scaleimage(v))
            ref.assert_equal(k + "/grad", g, lambda: R.gradients(v))
            ref.assert_equal(k + "/hess", h, lambda: R.hessian(v))
    a, b = stereo_view.shading_inputs(sc.images[0])
    ref.assert_equal("shading/img", a, lambda: R.shading()[0])
    ref.assert_equal("shading/grad", b, lambda: R.shading()[1])
    # Mi / ti, flen as the reference computes them (fp32, widened)
    wl = workload.build_workload(160, 120, 1, scale=2, scene=sc, shading=True)
    ref.assert_equal("Mi", wl.Mi, lambda: R.Mt()[0])
    ref.assert_equal("ti", wl.ti, lambda: R.Mt()[1])
    ref.assert_equal("flen", [wl.flen_px, wl.inv_flen],
                     lambda: [R.flen(0), R.inverse_flen(0)])
    if R:
        R.close()


def test_set_scale_mirror_colour_views_bitwise():
    """Three-channel views: channel-wise blur, luminance of the blurred image
    (lib/stereo_view.cc:48-62) -- the numpy restatement against the compiled
    reference, all three outputs bitwise."""
    from util_scene import RefOutputs, colour_scene
    ref = RefOutputs("set_scale_mirror_colour")
    sc = colour_scene(160, 120, 1, 3)
    R = oref.RefScene(sc) if ref.live else None
    for scale in (1, 3):
        if R:
            R.set_scale(scale)
        for v in (0, 1):
            b, g, h = stereo_view.set_scale(sc.images[v], scale)
            assert b.shape == (120, 160, 3)
            k = f"s{scale}v{v}"
            ref.assert_equal(k + "/blur", b, lambda: R.scaleimage(v))
            ref.assert_equal(k + "/grad", g, lambda: R.gradients(v))
            ref.assert_equal(k + "/hess", h, lambda: R.hessian(v))
    if R:
        R.close()


@pytest.mark.skipif(not oref.available(), reason="oracle/_ref not built")
def test_reference_optimize_without_sgm_grows_from_the_features():
    """The oracle's use_sgm = false entry (ref_optimize_nosgm): the sparse depth
    Surface::create makes of the bundle holds the features, and optimize()
    grows a surface from them that lies on the scene's true surface."""
    from util_scene import colour_scene
    sc = colour_scene(320, 240, 2, 4)
    rng = np.random.default_rng(4)
    x, y = rng.integers(8, 312, 150), rng.integers(8, 232, 150)
    d = sc.true_depth[y, x].astype(np.float64)
    f = float(sc.flen[0]) * 320
    feats = np.stack([(x + 0.5 - 160) / f * d, (y + 0.5 - 120) / f * d, d], axis=1)
    R = oref.RefScene(sc)
    sparse, depth, normals = R.optimize_nosgm(feats, num_iterations=3, min_scale=3)
    R.close()
    hit = sparse[y, x]
    assert (hit > 0).all() and np.abs(hit - d).max() < 1e-3 * d.max()
    assert (sparse > 0).sum() <= 150
    m = depth > 0
    assert m.mean() > 0.05
    assert np.median(np.abs(depth[m] - sc.true_depth[m]) / sc.true_depth[m]) < 5e-3


@pytest.mark.skipif(not oref.available(), reason="oracle/_ref not built")
def test_surface_grid_matches_reference():
    for (w, h, scale) in ((640, 480, 2), (640, 480, 4), (417, 311, 3), (1920, 1080, 5)):
        sc = synth.make_scene(w, h, 1, seed_index=1) if w < 1000 else None
        if sc is None:
            continue
        R = oref.RefScene(sc)
        R.surface_create(scale, sc.init_depth)
        i = R.surface_info()
        ps, npx, npy, sx, sy = synth.surface_grid(w, h, scale)
        assert (i["patchsize"], i["npx"], i["npy"], i["start_x"], i["start_y"]) == \
            (ps, npx, npy, sx, sy)
        R.close()


def test_workload_restrict_keeps_csr_consistent():
    wl = workload.build_workload(256, 192, 3, scale=2, seed_index=1)
    sub = wl.restrict(5, 4, 10, 8)
    assert sub.patch_valid.sum() <= 80 and sub.patch_valid.sum() > 0
    assert sub.vis_off[-1] == len(sub.vis_ids)
    pv = sub.patch_valid.reshape(sub.npy, sub.npx)
    assert pv[:4].sum() == 0 and pv[:, :5].sum() == 0
    cnt = np.diff(sub.vis_off.astype(np.int64))
    assert np.all(cnt[sub.patch_valid == 0] == 0)
    full_cnt = np.diff(wl.vis_off.astype(np.int64))
    assert np.array_equal(cnt[sub.patch_valid != 0], full_cnt[sub.patch_valid != 0])
    # every node of a valid patch is valid
    nv = sub.node_valid.reshape(sub.npy + 1, sub.npx + 1)
    ys, xs = np.nonzero(pv)
    assert nv[ys, xs].all() and nv[ys + 1, xs + 1].all()


def test_round_robin_sharding():
    got = [sharding.views_of_rank(32, r, 8) for r in range(8)]
    assert all(len(g) == 4 for g in got)
    assert sorted(sum(got, [])) == list(range(32))
    assert sharding.views_of_rank(3, 5, 8) == []


def _gloo_worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    views = sharding.views_of_rank(5, rank, world)
    pix, secs = sharding.reduce_job_stats(100.0 * len(views), 1.0 + rank)
    Ab = np.full(272, float(rank + 1))
    tot = sharding.allreduce_lighting_normal_equations(Ab)
    if rank == 0:
        out.put((pix, secs, float(tot[0]), float(tot[271])))
    dist.destroy_process_group()


def test_gloo_world_size_2():
    """The N > 1 path on CPU: view sharding, job statistics (sum of work, max
    of time) and the opt-in lighting reduction over a 2-rank gloo group."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert res == (500.0, 2.0, 3.0, 3.0)


def test_expf_twin_matches_libm():
    """The device bilateral filter evaluates expf the way glibc does (table +
    cubic in double, one rounding); its host twin must give libm's bits."""
    import ctypes as C
    L = api.lib()
    L.smvsb_debug_expf.restype = C.c_float
    L.smvsb_debug_expf.argtypes = [C.c_float]
    libm = C.CDLL("libm.so.6")
    libm.expf.restype = C.c_float
    libm.expf.argtypes = [C.c_float]
    rng = np.random.default_rng(7)
    xs = np.concatenate([-(rng.random(20000) ** 2 * 50).astype(np.float32),
                         np.float32([-0.0, -1e-7, -1.0, -50.0, -86.9])])
    for x in xs:
        assert L.smvsb_debug_expf(float(x)) == libm.expf(float(x))


@pytest.mark.skipif(not oref.available(), reason="oracle/_ref not built")
def test_bench_reference_arm_prints_the_contract_line():
    """bench.py --impl reference needs no GPU: one short step must end with one
    JSON line carrying the contract's keys (metric, value, unit, impl,
    cpu_baseline, e2e with zero transfer bytes)."""
    import json
    import subprocess
    env = dict(os.environ, SMVSB_REF_THREADS="2")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl",
                          "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, env=env, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"].startswith("Gauss-Newton")
    assert line["value"] > 0 and line["unit"] == "Mpix-iters/s"
    assert line["cpu_baseline"]["kind"] == "reference" and line["cpu_baseline"]["cores"] == 2
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["higher_is_better"] is True and line["scaling"] == "weak"
