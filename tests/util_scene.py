"""Shared helpers of the parity tests: drive the compiled-verbatim reference
(oracle/_ref) and the CUDA library (through the C ABI) with identical arrays.

The oracle is used here only as the checker."""
from __future__ import annotations

import atexit
import hashlib
import os

import numpy as np

from smvs_b200 import api, synth
from oracle import ref as oref

REF_OUTPUTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden",
                           "ref_outputs.npz")
_recorded = {}


def _digest(a):
    """SHA-256 of an array's shape and values (integers widened to int64,
    floats to float64, -0 as 0): equal digests <=> np.array_equal."""
    a = np.asarray(a)
    if a.dtype.kind == "f":
        a = np.where(np.isnan(a), np.nan, a.astype(np.float64) + 0.0)
    else:
        a = a.astype(np.int64)
    h = hashlib.sha256(repr(a.shape).encode())
    h.update(np.ascontiguousarray(a).tobytes())
    return np.frombuffer(h.digest(), np.uint8)


def _write_recorded(path):
    old = dict(np.load(REF_OUTPUTS)) if os.path.exists(REF_OUTPUTS) else {}
    old.update(_recorded)
    np.savez_compressed(path, **old)


class RefOutputs:
    """What a test compares against the compiled reference: computed live when
    oracle/_ref is built, else read from tests/golden/ref_outputs.npz. Large
    outputs are stored as digests, which is all a comparison for equality
    needs. SMVSB_RECORD_REF=<file> writes the live values of a run, merged with
    the stored ones, to <file> (regenerate the fixture after a change of the
    inputs of these tests)."""

    def __init__(self, test):
        self.test = test
        self.live = oref.available()
        self.stored = None
        if not self.live:
            if not os.path.exists(REF_OUTPUTS):
                raise RuntimeError(f"neither oracle/_ref nor {REF_OUTPUTS}")
            self.stored = np.load(REF_OUTPUTS)
        rec = os.environ.get("SMVSB_RECORD_REF")
        if self.live and rec and not _recorded:
            atexit.register(_write_recorded, rec)

    def _key(self, key):
        return f"{self.test}/{key}"

    def array(self, key, fn):
        """A small reference output the test uses as an input: stored whole."""
        if not self.live:
            return self.stored[self._key(key)]
        a = np.asarray(fn())
        if os.environ.get("SMVSB_RECORD_REF"):
            _recorded[self._key(key)] = a
        return a

    def assert_equal(self, key, out, fn):
        """out equals the reference's output fn() element for element."""
        if not self.live:
            assert np.array_equal(_digest(out), self.stored[self._key(key) + "#sha256"]), key
            return
        ref = fn()
        assert np.array_equal(out, ref), key
        if os.environ.get("SMVSB_RECORD_REF"):
            _recorded[self._key(key) + "#sha256"] = _digest(ref)


def colour_scene(width, height, n_sub, seed_index, shading=False):
    """Three different channels per view (the NCC filter works on colour)."""
    import copy
    sc = synth.make_scene(width, height, n_sub, seed_index=seed_index, shading=shading)
    col = copy.copy(sc)
    rng = np.random.default_rng(seed_index)
    imgs = []
    for im in sc.images:
        f = im.astype(np.float32)
        chans = [np.clip(f * g + o + rng.normal(0, 2.0, f.shape), 0, 255)
                 for g, o in ((1.0, 0.0), (0.8, 20.0), (1.1, -10.0))]
        imgs.append(np.stack(chans, axis=2).astype(np.uint8))
    col.images = imgs
    return col


class Pair:
    """Reference scene + (optionally) a GPU context fed with the reference's
    own prepared arrays at one scale."""

    def __init__(self, width, height, n_sub, scale, seed_index=0, shading=False,
                 gpu=True, init_noise=0.02):
        self.scene = synth.make_scene(width, height, n_sub, seed_index=seed_index,
                                      shading=shading, init_noise=init_noise)
        self.R = oref.RefScene(self.scene, init_linear=shading)
        self.scale = scale
        self.R.set_scale(scale)
        if scale == 0:
            # a scale-0 surface only ever arises by subdividing a scale-1 one
            # (initialize_node_from_depth has an empty window at patch size 1)
            self.R.surface_create(1, self.scene.init_depth)
            self.R.surface_subdivide()
        else:
            self.R.surface_create(scale, self.scene.init_depth)
        self.R.compute_visibility()
        self.info = self.R.surface_info()
        self.nodes, self.node_valid, self.patch_valid = self.R.surface_get()
        self.vis_off, self.vis_ids = self.R.get_visibility()
        self.Mi, self.ti = self.R.Mt()
        self.ctx = None
        if gpu:
            self.ctx = api.Context(0)
            self.push_views()
            self.push_surface()

    def push_views(self):
        R, n = self.R, self.scene.n_sub
        sh_img, sh_grad = R.shading() if self.scene.shading else (None, None)
        self.ctx.set_views(R.gradients(0),
                           [R.gradients(k + 1) for k in range(n)],
                           [R.hessian(k + 1) for k in range(n)],
                           self.Mi, self.ti, R.flen(0), R.inverse_flen(0),
                           sh_img, sh_grad)

    def push_surface(self, nodes=None):
        i = self.info
        self.ctx.set_surface(i["scale"], i["npx"], i["npy"], i["start_x"],
                             i["start_y"], self.nodes if nodes is None else nodes,
                             self.node_valid, self.patch_valid, self.vis_off,
                             self.vis_ids)

    def close(self):
        if self.ctx is not None:
            self.ctx.close()
        self.R.close()


def bsc_to_dict(sysd):
    """{(block_row, block_col): 4x4} from the reference BSC arrays."""
    out = {}
    outer, inner, vals = sysd["Houter"], sysd["Hinner"], sysd["Hvals"]
    for col in range(len(outer) - 1):
        for k in range(int(outer[col]), int(outer[col + 1])):
            out[(int(inner[k]) // 4, col)] = vals[k].reshape(4, 4)
    return out


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))
