"""ctypes binding of oracle/_ref/libsmvs_ref.so -- the reference's own
hot-path sources compiled verbatim against the MVE shim (oracle/Makefile).

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_ref", "libsmvs_ref.so")

# The same C driver (oracle/ref_driver.cc) is also linked into
# _ref/integration/libsmvs_ref_b200.so, where the reference's host code runs
# with the GPU hot path patched in (integration/Makefile). It sits under _ref/
# so that it goes wherever the reference build goes.
INTEGRATION_LIB_PATH = os.path.join(_HERE, "_ref", "integration", "libsmvs_ref_b200.so")
_libs = {}


def available() -> bool:
    return os.path.exists(LIB_PATH)


def load(path=None):
    path = path or LIB_PATH
    if path not in _libs:
        if not os.path.exists(path):
            raise RuntimeError(f"{path} not built (run `make -C oracle ref` / "
                               "`make -C integration` where /root/reference exists)")
        L = C.CDLL(path)
        L.ref_scene_create.restype = C.c_void_p
        L.ref_view_get_flen.restype = C.c_float
        L.ref_view_get_inverse_flen.restype = C.c_float
        L.ref_gn_construct.restype = C.c_int64
        L.ref_get_visibility.restype = C.c_uint64
        _libs[path] = L
    return _libs[path]


def lib():
    return load(None)


def _p(a, t=None):
    if a is None:
        return None
    return a.ctypes.data_as(C.c_void_p)


class RefScene:
    """The reference's StereoViews + DepthOptimizer over a synthetic scene."""

    def __init__(self, scene, init_linear=False, lib_path=None):
        L = self.L = load(lib_path)
        n = 1 + scene.n_sub
        self.scene = scene
        self.n_sub = scene.n_sub
        self.w, self.h = scene.width, scene.height
        imgs = [np.ascontiguousarray(im) for im in scene.images]
        self._keep = imgs
        ws = (C.c_int * n)(*[im.shape[1] for im in imgs])
        hs = (C.c_int * n)(*[im.shape[0] for im in imgs])
        chs = (C.c_int * n)(*[1 if im.ndim == 2 else im.shape[2] for im in imgs])
        ptrs = (C.c_void_p * n)(*[im.ctypes.data for im in imgs])
        flen = np.ascontiguousarray(scene.flen, dtype=np.float32)
        rot = np.ascontiguousarray(scene.rot, dtype=np.float32)
        trans = np.ascontiguousarray(scene.trans, dtype=np.float32)
        self.h_ = C.c_void_p(L.ref_scene_create(n, ws, hs, chs, ptrs, _p(flen),
                                                _p(rot), _p(trans), int(init_linear)))

    def close(self):
        if self.h_:
            self.L.ref_scene_destroy(self.h_)
            self.h_ = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- views ---------------------------------------------------------
    def set_scale(self, scale):
        self.L.ref_scene_set_scale(self.h_, int(scale))

    def gradients(self, v):
        out = np.empty((self.h, self.w, 2), dtype=np.float32)
        self.L.ref_view_get_gradients(self.h_, v, _p(out))
        return out

    def hessian(self, v):
        out = np.empty((self.h, self.w, 3), dtype=np.float32)
        self.L.ref_view_get_hessian(self.h_, v, _p(out))
        return out

    def scaleimage(self, v):
        """StereoView::get_scaleimage(): the blurred image with all its channels."""
        im = self.scene.images[v]
        ch = 1 if im.ndim == 2 else im.shape[2]
        out = np.empty((self.h, self.w, ch), dtype=np.float32)
        self.L.ref_view_get_scaleimage(self.h_, v, _p(out))
        return out[:, :, 0] if ch == 1 else out

    def shading(self):
        img = np.empty((self.h, self.w), dtype=np.float32)
        grad = np.empty((self.h, self.w, 2), dtype=np.float32)
        if self.L.ref_view_get_shading(self.h_, _p(img), _p(grad)) != 0:
            return None, None
        return img, grad

    def set_arrays(self, v, grad, hess):
        grad = np.ascontiguousarray(grad, dtype=np.float32)
        hess = None if hess is None else np.ascontiguousarray(hess, dtype=np.float32)
        self.L.ref_view_set_arrays(self.h_, v, _p(grad), _p(hess))

    def set_shading(self, img, grad):
        img = np.ascontiguousarray(img, dtype=np.float32)
        grad = np.ascontiguousarray(grad, dtype=np.float32)
        self.L.ref_view_set_shading(self.h_, _p(img), _p(grad))

    def flen(self, v=0):
        return float(self.L.ref_view_get_flen(self.h_, v))

    def inverse_flen(self, v=0):
        return float(self.L.ref_view_get_inverse_flen(self.h_, v))

    def Mt(self):
        Mi = np.empty((self.n_sub, 9), dtype=np.float64)
        ti = np.empty((self.n_sub, 3), dtype=np.float64)
        self.L.ref_scene_get_Mt(self.h_, _p(Mi), _p(ti))
        return Mi, ti

    # -- surface -------------------------------------------------------
    def surface_create(self, scale, init_depth):
        d = np.ascontiguousarray(init_depth, dtype=np.float32)
        self.L.ref_surface_create(self.h_, int(scale), _p(d))

    def surface_info(self):
        info = (C.c_int * 6)()
        self.L.ref_surface_info(self.h_, info)
        return dict(scale=info[0], npx=info[1], npy=info[2], start_x=info[3],
                    start_y=info[4], patchsize=info[5])

    def surface_get(self):
        i = self.surface_info()
        nn = (i["npx"] + 1) * (i["npy"] + 1)
        npatch = i["npx"] * i["npy"]
        nodes = np.empty((nn, 4), dtype=np.float64)
        nv = np.empty(nn, dtype=np.uint8)
        pv = np.empty(npatch, dtype=np.uint8)
        self.L.ref_surface_get(self.h_, _p(nodes), _p(nv), _p(pv))
        return nodes, nv, pv

    def surface_set(self, nodes, node_valid, patch_valid):
        nodes = np.ascontiguousarray(nodes, dtype=np.float64)
        nv = np.ascontiguousarray(node_valid, dtype=np.uint8)
        pv = np.ascontiguousarray(patch_valid, dtype=np.uint8)
        self.L.ref_surface_set(self.h_, _p(nodes), _p(nv), _p(pv))

    def surface_subdivide(self):
        self.L.ref_surface_subdivide(self.h_)

    def surface_fill_from_depth(self):
        self.L.ref_surface_fill_from_depth(self.h_)

    def surface_remove_isolated(self):
        self.L.ref_surface_remove_isolated(self.h_)

    def surface_expand(self):
        return int(self.L.ref_surface_expand(self.h_))

    def surface_depth(self):
        out = np.empty((self.h, self.w), dtype=np.float32)
        self.L.ref_surface_get_depth(self.h_, _p(out))
        return out

    def surface_normals(self):
        out = np.empty((self.h, self.w, 3), dtype=np.float32)
        self.L.ref_surface_get_normals(self.h_, _p(out))
        return out

    def node_derivative_table(self):
        ps = self.surface_info()["patchsize"]
        out = np.empty((ps * ps, 96), dtype=np.float64)
        self.L.ref_node_derivative_table(self.h_, _p(out))
        return out

    # -- visibility ----------------------------------------------------
    def compute_visibility(self):
        return int(self.L.ref_compute_visibility(self.h_))

    def create_subview_surfaces(self, use_sgm=True):
        """DepthOptimizer::create_subview_surfaces alone; returns patches left."""
        return int(self.L.ref_create_subview_surfaces(self.h_, int(bool(use_sgm))))

    def cut_boundaries(self):
        """One DepthOptimizer::cut_boundaries(); returns patches deleted."""
        return int(self.L.ref_cut_boundaries(self.h_))

    def set_sgm_depth(self, depth):
        d = np.ascontiguousarray(depth, dtype=np.float32)
        self.L.ref_set_sgm_depth(self.h_, d.ctypes.data_as(C.c_void_p))

    def inverse_calibration(self):
        out = np.empty(9, dtype=np.float32)
        self.L.ref_main_inverse_calibration(self.h_, out.ctypes.data_as(C.c_void_p))
        return out

    def bilateral_filter(self, depth):
        """DepthOptimizer::depthmap_bilateral_filter(depth, main image)."""
        d = np.ascontiguousarray(depth, dtype=np.float32)
        out = np.empty((self.h, self.w), dtype=np.float32)
        self.L.ref_bilateral_filter(self.h_, _p(d), d.shape[1], d.shape[0], _p(out))
        return out

    def image(self, v):
        """StereoView::get_image(): the unblurred float image of view v."""
        ch = int(self.L.ref_view_get_image(self.h_, v, None))
        h, w = self.scene.images[v].shape[:2]
        out = np.empty((h, w, ch), dtype=np.float32)
        self.L.ref_view_get_image(self.h_, v, _p(out))
        return out[:, :, 0] if ch == 1 else out

    def get_visibility(self):
        i = self.surface_info()
        npatch = i["npx"] * i["npy"]
        off = np.empty(npatch + 1, dtype=np.uint32)
        total = int(self.L.ref_get_visibility(self.h_, _p(off), None))
        ids = np.empty(max(total, 1), dtype=np.uint8)
        self.L.ref_get_visibility(self.h_, _p(off), _p(ids))
        return off, ids[:total]

    def set_visibility(self, off, ids):
        off = np.ascontiguousarray(off, dtype=np.uint32)
        ids = np.ascontiguousarray(ids, dtype=np.uint8)
        self._vis_keep = (off, ids)
        self.L.ref_set_visibility(self.h_, _p(off), _p(ids))

    # -- Gauss-Newton --------------------------------------------------
    def gn_construct(self, active, light16=None, regularization=0.01,
                     light_surf_regularization=0.0):
        active = np.ascontiguousarray(active, dtype=np.uint8)
        l = None if light16 is None else np.ascontiguousarray(light16, dtype=np.float64)
        return int(self.L.ref_gn_construct(self.h_, _p(active), _p(l),
                                          C.c_double(regularization),
                                          C.c_double(light_surf_regularization)))

    def get_system(self):
        sz = (C.c_uint64 * 3)()
        self.L.ref_get_system_sizes(self.h_, sz)
        n, nh, npc = int(sz[0]), int(sz[1]), int(sz[2])
        g = np.empty(n, dtype=np.float64)
        Hv = np.empty((nh, 16), dtype=np.float64)
        Ho = np.empty(n // 4 + 1, dtype=np.uint64)
        Hi = np.empty(nh, dtype=np.uint64)
        Pv = np.empty((npc, 16), dtype=np.float64)
        Po = np.empty(n // 4 + 1, dtype=np.uint64)
        Pi = np.empty(npc, dtype=np.uint64)
        self.L.ref_get_system(self.h_, _p(g), _p(Hv), _p(Ho), _p(Hi), _p(Pv), _p(Po), _p(Pi))
        return dict(g=g, Hvals=Hv, Houter=Ho, Hinner=Hi, Pvals=Pv, Pouter=Po, Pinner=Pi)

    def hessian_multiply(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.empty_like(x)
        self.L.ref_hessian_multiply(self.h_, _p(x), _p(y))
        return y

    def cg_solve(self, max_iter=200, err_tol=-1.0, q_tol=1e-3):
        sz = (C.c_uint64 * 3)()
        self.L.ref_get_system_sizes(self.h_, sz)
        x = np.empty(int(sz[0]), dtype=np.float64)
        it, info = C.c_int(0), C.c_int(0)
        self.L.ref_cg_solve(self.h_, int(max_iter), C.c_double(err_tol),
                           C.c_double(q_tol), _p(x), C.byref(it), C.byref(info))
        return x, it.value, info.value

    def update_nodes(self, delta, active, reproj_thresh=0.15, full_opt=False):
        delta = np.ascontiguousarray(delta, dtype=np.float64)
        act = np.array(active, dtype=np.uint8, copy=True)
        n_active = C.c_uint64(0)
        mean_shift = C.c_double(0)
        self.L.ref_update_nodes(self.h_, _p(delta), C.c_double(reproj_thresh),
                               int(full_opt), _p(act), C.byref(n_active),
                               C.byref(mean_shift))
        return act, int(n_active.value), float(mean_shift.value)

    def newton_loop(self, light16=None, regularization=0.01,
                    light_surf_regularization=0.0, max_steps=200):
        l = None if light16 is None else np.ascontiguousarray(light16, dtype=np.float64)
        st = np.zeros(8, dtype=np.float64)
        self.L.ref_newton_loop(self.h_, _p(l), C.c_double(regularization),
                              C.c_double(light_surf_regularization), int(max_steps), _p(st))
        return dict(newton_steps=int(st[0]), cg_iterations=int(st[1]),
                    pixel_iterations=float(st[2]), t_construct=float(st[3]),
                    t_solve=float(st[4]), t_update=float(st[5]),
                    n_active=int(st[6]), nan=bool(st[7]))

    def fit_lighting(self):
        p = np.zeros(16, dtype=np.float64)
        if self.L.ref_fit_lighting(self.h_, _p(p)) != 0:
            return None
        return p

    def optimize(self, sgm_depth, regularization=0.01, num_iterations=5,
                 min_scale=2, use_shading=False, debug_lvl=0):
        d = np.ascontiguousarray(sgm_depth, dtype=np.float32)
        depth = np.empty((self.h, self.w), dtype=np.float32)
        normals = np.empty((self.h, self.w, 3), dtype=np.float32)
        light = np.zeros(16, dtype=np.float64)
        self.L.ref_optimize(self.h_, _p(d), C.c_double(regularization),
                           int(num_iterations), int(min_scale), int(use_shading),
                           int(debug_lvl), _p(depth), _p(normals), _p(light))
        return depth, normals, light

    def optimize_nosgm(self, features, regularization=0.01, num_iterations=5, min_scale=2):
        """DepthOptimizer::optimize() with use_sgm = false: `features` (n, 3)
        world points the main view observes (the bundle). Returns (sparse
        initial depth as Surface::create makes it, depth, normals)."""
        f = np.ascontiguousarray(features, dtype=np.float32)
        sparse = np.empty((self.h, self.w), dtype=np.float32)
        depth = np.empty((self.h, self.w), dtype=np.float32)
        normals = np.empty((self.h, self.w, 3), dtype=np.float32)
        self.L.ref_optimize_nosgm(self.h_, int(f.shape[0]), _p(f), C.c_double(regularization),
                                  int(num_iterations), int(min_scale), _p(sparse), _p(depth),
                                  _p(normals))
        return sparse, depth, normals

    def sgm_roundtrip(self, depth):
        """StereoView::get_sgm_depth() of a depth stored as "smvs-sgm"."""
        d = np.ascontiguousarray(depth, dtype=np.float32)
        out = np.empty((self.h, self.w), dtype=np.float32)
        self.L.ref_sgm_roundtrip(self.h_, _p(d), _p(out))
        return out

    # -- SGM -------------------------------------------------------------
    def sgm_dims(self, v, scale):
        info = (C.c_int * 2)()
        self.L.ref_sgm_dims(self.h_, v, scale, info)
        return info[0], info[1]

    def sgm_run(self, a, b, scale, num_steps, min_depth, max_depth,
                penalty1=6, penalty2=96, volumes=False):
        w, h = self.sgm_dims(a, scale)
        depth = np.empty((h, w), dtype=np.float32)
        cost = np.empty((h, w, num_steps), dtype=np.uint16) if volumes else None
        sgm = np.empty((h, w, num_steps), dtype=np.uint16) if volumes else None
        times = np.zeros(3, dtype=np.float64)
        self.L.ref_sgm_run(self.h_, a, b, scale, num_steps, C.c_float(min_depth),
                          C.c_float(max_depth), penalty1, penalty2, _p(depth),
                          _p(cost), _p(sgm), _p(times))
        return dict(depth=depth, cost=cost, sgm=sgm, times=times)

    def sgm_reconstruct(self, a, b, scale, num_steps, min_depth, max_depth):
        w, h = self.sgm_dims(a, scale)
        depth = np.empty((h, w), dtype=np.float32)
        self.L.ref_sgm_reconstruct(self.h_, a, b, scale, num_steps,
                                  C.c_float(min_depth), C.c_float(max_depth), _p(depth))
        return depth

    def reprojection(self, a, b, aw, ah, bw, bh):
        M = np.empty(9, dtype=np.float32)
        t = np.empty(3, dtype=np.float32)
        self.L.ref_reprojection(self.h_, a, b, aw, ah, bw, bh, _p(M), _p(t))
        return M, t


# ---------------------------------------------------------------------------
# unit-level entry points (the reference's own known-answer tests run on them)
# ---------------------------------------------------------------------------

def cut_depth_maps(flen, rot, trans, depths, normals, run=True, lib_path=None):
    """MeshGenerator::cut_depth_maps of the compiled reference on n views:
    cameras (flen (n,), world-to-camera rot (n, 9), trans (n, 3)), depth maps in
    MVE convention, world-space normal maps. Returns (cut maps or None,
    invproj (n, 9), cam_to_world (n, 16), KR (n, 9), t (n, 3)). lib_path =
    INTEGRATION_LIB_PATH runs the drop-in member (integration/b200_mesh_generator.cc)."""
    n = len(depths)
    d = [np.ascontiguousarray(a, dtype=np.float32) for a in depths]
    nr = [np.ascontiguousarray(a, dtype=np.float32) for a in normals]
    outs = [np.empty_like(a) for a in d]
    w = (C.c_int * n)(*[a.shape[1] for a in d])
    h = (C.c_int * n)(*[a.shape[0] for a in d])
    dp = (C.c_void_p * n)(*[a.ctypes.data for a in d])
    npp = (C.c_void_p * n)(*[a.ctypes.data for a in nr])
    op = (C.c_void_p * n)(*[a.ctypes.data for a in outs])
    fl = np.ascontiguousarray(flen, dtype=np.float32)
    ro = np.ascontiguousarray(rot, dtype=np.float32).reshape(n, 9)
    tr = np.ascontiguousarray(trans, dtype=np.float32).reshape(n, 3)
    inv = np.empty((n, 9), np.float32)
    ctw = np.empty((n, 16), np.float32)
    KR = np.empty((n, 9), np.float32)
    t = np.empty((n, 3), np.float32)
    load(lib_path).ref_cut_depth_maps(n, w, h, _p(fl), _p(ro), _p(tr), dp, npp, op if run else None,
                                      _p(inv), _p(ctw), _p(KR), _p(t))
    return (outs if run else None), inv, ctw, KR, t


class Units:
    """Per-function access to the compiled reference (BicubicPatch,
    Correspondence, surfderiv, sh, ldl_inverse)."""

    name = "reference (oracle/_ref)"

    @staticmethod
    def bicubic_eval(nodes16, x, y):
        n = np.ascontiguousarray(nodes16, dtype=np.float64).reshape(16)
        out = np.empty(6, dtype=np.float64)
        lib().ref_bicubic_eval(_p(n), C.c_double(x), C.c_double(y), _p(out))
        return out

    @staticmethod
    def node_derivatives(x, y, patchsize=0.0):
        out = np.empty(96, dtype=np.float64)
        lib().ref_bicubic_node_derivatives(C.c_double(x), C.c_double(y),
                                           C.c_double(patchsize), _p(out))
        return out

    @staticmethod
    def correspondence(M, t, u, v, w, wx=0.0, wy=0.0, grad=(0.0, 0.0), dn=None):
        M = np.ascontiguousarray(M, dtype=np.float64).reshape(9)
        t = np.ascontiguousarray(t, dtype=np.float64).reshape(3)
        g = np.ascontiguousarray(grad, dtype=np.float64).reshape(2)
        dn = np.zeros(96) if dn is None else np.ascontiguousarray(dn, dtype=np.float64)
        proj = np.empty(2); jac = np.empty(4); c_dn = np.empty((16, 2)); j_dn = np.empty((16, 2))
        depth = C.c_double(0)
        lib().ref_correspondence(_p(M), _p(t), C.c_double(u), C.c_double(v), C.c_double(w),
                                 C.c_double(wx), C.c_double(wy), _p(g), _p(dn), _p(proj),
                                 _p(jac), _p(c_dn), _p(j_dn), C.byref(depth))
        return dict(proj=proj, jac=jac, c_dn=c_dn, jac_dn=j_dn, depth=depth.value)

    @staticmethod
    def surface_derivatives(dn, x, y, f, w, dx, dy, dxy, dxx, dyy):
        dn = np.ascontiguousarray(dn, dtype=np.float64)
        normal = np.empty(3); div = np.empty(6); dd = np.empty(96); nd = np.empty(48)
        lib().ref_surface_derivatives(_p(dn), *[C.c_double(a) for a in
                                                (x, y, f, w, dx, dy, dxy, dxx, dyy)],
                                      _p(normal), _p(div), _p(dd), _p(nd))
        return dict(normal=normal, div=div, div_deriv=dd, normal_deriv=nd)

    @staticmethod
    def sh_4band(normal):
        n = np.ascontiguousarray(normal, dtype=np.float64)
        sh = np.empty(16); d = np.empty(48)
        lib().ref_sh_4band(_p(n), _p(sh), _p(d))
        return sh, d

    @staticmethod
    def ldl_inverse(A):
        A = np.array(A, dtype=np.float64, copy=True)
        n = A.shape[0]
        lib().ref_ldl_inverse(_p(A), n)
        return A


    # -- tests/gtest_matrix_vector.cc:33-356 ---------------------------------
    has_linear_algebra = True

    @staticmethod
    def ssevector(op, a, b=None, factor=0.0):
        ops = dict(dot=0, add=1, subtract=2, multiply=3, multiply_add=4, multiply_sub=5)
        a = np.ascontiguousarray(a, dtype=np.float64)
        bb = None if b is None else np.ascontiguousarray(b, dtype=np.float64)
        out = np.empty(1 if op == "dot" else len(a), dtype=np.float64)
        lib().ref_ssevector_op(ops[op], len(a), _p(a), _p(bb), C.c_double(factor), _p(out))
        return float(out[0]) if op == "dot" else out

    @staticmethod
    def bsm2(dim, blocks=None, triplets=None, invert=False, x=None):
        """BlockSparseMatrix<2>: (num_non_zero, A x)."""
        blocks = blocks or []
        triplets = triplets or []
        brc = np.array([[r, c] for r, c, _ in blocks], dtype=np.int32).reshape(-1)
        bv = np.array([v for _, _, v in blocks], dtype=np.float64).reshape(-1)
        trc = np.array([[r, c] for r, c, _ in triplets], dtype=np.int32).reshape(-1)
        tv = np.array([v for _, _, v in triplets], dtype=np.float64)
        xv = None if x is None else np.ascontiguousarray(x, dtype=np.float64)
        y = None if x is None else np.empty(dim, dtype=np.float64)
        nnz = lib().ref_bsm2(dim, len(blocks), _p(brc) if len(brc) else None,
                             _p(bv) if len(bv) else None, len(triplets),
                             _p(trc) if len(trc) else None, _p(tv) if len(tv) else None,
                             int(invert), _p(xv), _p(y))
        return int(nnz), y
