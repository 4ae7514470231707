#!/usr/bin/env python
"""Generate tests/golden/*.npz by EXECUTING the reference's own python source.

Run in the build container only (needs /root/reference):

    python tests/golden/make_golden.py

The reference (openai/iaf) is python-2 + Theano/TensorFlow and cannot be imported
here (SURVEY F4).  What this script does instead:

 1. reads the reference's source files from /root/reference,
 2. makes them parseable by python 3 WITHOUT touching their logic: ``print x`` ->
    ``print(x)``, ``map(...)`` -> ``list(map(...))``, and every ``a / b`` becomes
    ``_py2div(a, b)`` (python-2 semantics: floor for two ints, true division otherwise),
 3. exec's them against a tiny numpy-backed stand-in for the handful of TF / Theano
    primitives they call.  The convolution primitive (cuDNN behind tf.nn.conv2d /
    dnn_conv) is stood in for by torch's CPU float64 conv2d -- an implementation that is
    independent of both the oracle (oracle/iaf_oracle.py) and the CUDA kernels.

Everything that is *the reference's algorithm* -- mask construction, weight
normalisation, layer order, where the context is added, zerodiagonal flags, the pad
channel, the 0.1 scaling and affine update inside IAFLayer.down, the free-bits KL --
is therefore run from the reference's own lines, in float64, on float32-valued
inputs.  Inputs are regenerated in the tests from seeds (oracle.make_params /
make_inputs use the legacy, version-stable np.random.RandomState); the fixtures
store the outputs plus input checksums.
"""
import ast
import contextlib
import os
import re
import sys
import types

import numpy as np
import torch

REF = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
from oracle import iaf_oracle as O  # noqa: E402  (only for make_params / make_inputs seeds)


# --------------------------------------------------------------------------
# python2 -> python3 source shims (syntax only)
# --------------------------------------------------------------------------
def _py2div(a, b):
    ints = (int, np.integer)
    if isinstance(a, ints) and isinstance(b, ints) and not isinstance(a, bool):
        return a // b
    return a / b


class _Div(ast.NodeTransformer):
    def visit_BinOp(self, node):
        self.generic_visit(node)
        if isinstance(node.op, ast.Div):
            return ast.copy_location(
                ast.Call(func=ast.Name(id="_py2div", ctx=ast.Load()), args=[node.left, node.right], keywords=[]),
                node)
        return node


def py2_compile(src, filename):
    src = re.sub(r"^(\s*)print\s+(?!\()(.*)$", r"\1print(\2)", src, flags=re.M)
    src = re.sub(r"(?<![\w.])map\(([^\n]*?)\)$", r"list(map(\1))", src, flags=re.M)
    tree = _Div().visit(ast.parse(src, filename))
    ast.fix_missing_locations(tree)
    return compile(tree, filename, "exec")


def read(path):
    with open(os.path.join(REF, path)) as f:
        return f.read()


def extract(src, start_pat, end_pat):
    """Text of src from the line matching start_pat up to (not incl.) the next line matching end_pat."""
    m = re.search(start_pat, src, flags=re.M)
    assert m, start_pat
    e = re.search(end_pat, src[m.end():], flags=re.M)
    return src[m.start(): m.end() + (e.start() if e else len(src))]


# --------------------------------------------------------------------------
# tensor stand-in
# --------------------------------------------------------------------------
class _Tag(object):
    def __init__(self, v):
        self.test_value = v


class _Shape(list):
    def as_list(self):
        return list(self)


class RT(np.ndarray):
    """ndarray that also answers the few Theano / TF tensor methods the reference uses."""

    def __new__(cls, a):
        return np.asarray(a, dtype=np.float64).view(cls)

    @property
    def tag(self):
        return _Tag(np.asarray(self))

    def dimshuffle(self, *pat):
        a = np.asarray(self)
        idx = [p for p in pat if p != "x"]
        a = a.transpose(idx) if idx else a
        shape, it = [], iter(a.shape)
        for p in pat:
            shape.append(1 if p == "x" else next(it))
        return RT(a.reshape(shape))

    def get_shape(self):
        return _Shape(self.shape)

    def initialized_value(self):
        return self

    def set_shape(self, shape):
        assert list(self.shape) == [int(v) for v in shape]


def conv_nchw(x, w_oihw, flip):
    """cuDNN stand-in: torch CPU float64.  flip=True -> true convolution."""
    w = torch.from_numpy(np.ascontiguousarray(np.asarray(w_oihw, dtype=np.float64)))
    if flip:
        w = torch.flip(w, dims=(2, 3))
    return torch.nn.functional.conv2d(torch.from_numpy(np.ascontiguousarray(np.asarray(x, dtype=np.float64))), w)


# --------------------------------------------------------------------------
# TensorFlow stand-in (TF <= 0.11 API as used by the reference)
# --------------------------------------------------------------------------
class TFShim(types.ModuleType):
    float32 = "float32"

    def __init__(self):
        super().__init__("tensorflow")
        self.store = {}
        self.scope = []
        self.noise = []  # queue of arrays returned by random_normal
        nn = types.SimpleNamespace()
        nn.elu = lambda x: RT(np.where(np.asarray(x) < 0, np.expm1(np.minimum(np.asarray(x), 0)), np.asarray(x)))
        nn.l2_normalize = self._l2n
        nn.conv2d = self._conv2d
        self.nn = nn

    # variables -----------------------------------------------------------
    @contextlib.contextmanager
    def variable_scope(self, name):
        self.scope.append(name)
        try:
            yield
        finally:
            self.scope.pop()

    def get_variable(self, name, shape=None, dtype=None, initializer=None):
        key = "/".join(self.scope + [name])
        v = self.store[key]
        if shape is not None:
            assert list(v.shape) == [int(s) for s in shape], (key, v.shape, shape)
        return RT(v)

    # primitives ------------------------------------------------------------
    @staticmethod
    def _l2n(x, dim, epsilon=1e-12):
        x = np.asarray(x)
        sq = np.sum(np.square(x), axis=tuple(dim), keepdims=True)
        return RT(x / np.sqrt(np.maximum(sq, epsilon)))

    @staticmethod
    def _conv2d(x, w, strides, pad, data_format="NHWC"):
        assert data_format == "NCHW" and pad == "SAME" and list(strides) == [1, 1, 1, 1]
        w = np.asarray(w)  # [kh,kw,ci,co]
        kh, kw = w.shape[:2]
        xp = np.pad(np.asarray(x), ((0, 0), (0, 0), ((kh - 1) // 2, kh // 2), ((kw - 1) // 2, kw // 2)))
        return RT(conv_nchw(xp, w.transpose(3, 2, 0, 1), flip=False).numpy())

    def constant(self, v):
        return RT(v)

    def exp(self, x):
        return RT(np.exp(np.asarray(x)))

    def log(self, x):
        return RT(np.log(np.asarray(x)))

    def square(self, x):
        return RT(np.square(np.asarray(x)))

    def reshape(self, x, shape):
        x = np.asarray(x)
        return x.reshape(shape) if x.dtype.kind in "iu" else RT(x.reshape(shape))

    def reduce_sum(self, x, axes=None, keep_dims=False):
        return RT(np.sum(np.asarray(x), axis=None if axes is None else tuple(axes), keepdims=keep_dims))

    def reduce_mean(self, x, axes=None, keep_dims=False):
        return RT(np.mean(np.asarray(x), axis=None if axes is None else tuple(axes), keepdims=keep_dims))

    def reduce_max(self, x, axes=None, keep_dims=False):
        return RT(np.max(np.asarray(x), axis=None if axes is None else tuple(axes), keepdims=keep_dims))

    def maximum(self, a, b):
        return RT(np.maximum(a, b))

    def tile(self, x, reps):
        x = np.asarray(x)
        return np.tile(x, reps) if x.dtype.kind in "iu" else RT(np.tile(x, reps))

    def concat(self, axis, values):  # TF<=0.12 argument order
        return RT(np.concatenate([np.asarray(v) for v in values], axis=axis))

    def zeros(self, shape):
        return RT(np.zeros(shape))

    def shape(self, x):
        return np.asarray(x).shape

    def random_normal(self, shape):
        e = self.noise.pop(0)
        assert tuple(e.shape) == tuple(shape)
        return RT(e)

    def slice(self, x, begin, size):
        x = np.asarray(x)
        idx = tuple(slice(int(b), None if int(s) == -1 else int(b) + int(s)) for b, s in zip(begin, size))
        return RT(x[idx])

    def range(self, n):
        return np.arange(n)

    def gather(self, x, idx):
        return RT(np.asarray(x)[np.asarray(idx)])


@contextlib.contextmanager
def _arg_scope(fns, **kw):
    assert not kw
    yield


def load_tf_reference():
    """exec tf_utils/layers.py + distributions.py + common.split + tf_train.IAFLayer."""
    tf = TFShim()
    fw = types.ModuleType("tensorflow.contrib.framework.python.ops")
    fw.arg_scope = _arg_scope
    fw.add_arg_scope = lambda f: f
    mods = {"tensorflow": tf, "tensorflow.contrib": types.ModuleType("c"),
            "tensorflow.contrib.framework": types.ModuleType("c"),
            "tensorflow.contrib.framework.python": types.ModuleType("c"),
            "tensorflow.contrib.framework.python.ops": fw}
    saved = {k: sys.modules.get(k) for k in mods}
    sys.modules.update(mods)
    try:
        layers = {"_py2div": _py2div}
        exec(py2_compile(read("tf_utils/layers.py"), "tf_utils/layers.py"), layers)
        dist = {"_py2div": _py2div}
        exec(py2_compile(read("tf_utils/distributions.py"), "tf_utils/distributions.py"), dist)
        common = {"_py2div": _py2div, "np": np, "tf": tf}
        exec(py2_compile(extract(read("tf_utils/common.py"), r"^def split\(", r"^def "), "tf_utils/common.py"), common)
        train = {"_py2div": _py2div, "np": np, "tf": tf, "arg_scope": _arg_scope,
                 "conv2d": layers["conv2d"], "deconv2d": layers["deconv2d"],
                 "ar_multiconv2d": layers["ar_multiconv2d"],
                 "resize_nearest_neighbor": layers["resize_nearest_neighbor"],
                 "DiagonalGaussian": dist["DiagonalGaussian"], "split": common["split"]}
        exec(py2_compile(extract(read("tf_train.py"), r"^class IAFLayer", r"^def get_default_hparams"),
                         "tf_train.py"), train)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    return tf, layers, dist, train


# --------------------------------------------------------------------------
# Theano / graphy stand-in
# --------------------------------------------------------------------------
def _root(a):
    while isinstance(a.base, np.ndarray):
        a = a.base
    return a


def load_theano_reference():
    T = types.ModuleType("theano.tensor")
    T.exp = lambda x: RT(np.exp(np.asarray(x)))
    T.sqrt = lambda x: RT(np.sqrt(np.asarray(x)))
    T.log = lambda x: RT(np.log(np.asarray(x)))
    T.tanh = lambda x: RT(np.tanh(np.asarray(x)))
    T.zeros = lambda shape, dtype=None: RT(np.zeros(tuple(int(s) for s in shape)))
    T.switch = lambda c, a, b: RT(np.where(c, a, b))
    T.maximum = lambda a, b: RT(np.maximum(a, b))

    def set_subtensor(sub, val):
        base = _root(sub)
        sub[...] = val
        return RT(base) if not isinstance(base, RT) else base
    T.set_subtensor = set_subtensor
    T.nnet = types.SimpleNamespace(softplus=lambda x: RT(np.logaddexp(0, np.asarray(x))),
                                   sigmoid=lambda x: RT(1 / (1 + np.exp(-np.asarray(x)))))

    class Struct:  # graphy/__init__.py:35-39; __call__ entry must be callable on the instance
        def __init__(self, **entries):
            self.__dict__.update(entries)

        def __call__(self, *a, **k):
            return self.__dict__["__call__"](*a, **k)

    G = types.ModuleType("graphy")
    G.floatX = "float64"
    G.sharedf = lambda x, **k: RT(np.asarray(x, dtype=np.float64))
    G.Struct = Struct

    theano = types.ModuleType("theano")
    theano.tensor = T
    N = types.ModuleType("graphy.nodes")
    Nconv = types.ModuleType("graphy.nodes.conv")
    N.conv = Nconv
    G.nodes = N

    def dnn_conv(h, kerns, border_mode="valid", conv_mode="conv"):
        assert border_mode == "valid"
        return RT(conv_nchw(h, kerns, flip=(conv_mode == "conv")).numpy())
    Nconv.dnn_conv = dnn_conv

    conv_src = read("graphy/nodes/conv.py")
    ns = {"_py2div": _py2div, "T": T, "G": G, "np": np}
    exec(py2_compile(extract(conv_src, r"^def pad2dwithchannel", r"^# Multi-scale conv"), "graphy/nodes/conv.py"), ns)
    Nconv.pad2dwithchannel = ns["pad2dwithchannel"]

    init_src = read("graphy/nodes/__init__.py")
    ns2 = {"_py2div": _py2div, "T": T, "G": G, "np": np}
    exec(py2_compile(extract(init_src, r"^def nonlinearity", r"^# n_in is an int"), "graphy/nodes/__init__.py"), ns2)
    N.nonlinearity = ns2["nonlinearity"]

    mods = {"theano": theano, "theano.tensor": T, "graphy": G, "graphy.nodes": N, "graphy.nodes.conv": Nconv}
    saved = {k: sys.modules.get(k) for k in mods}
    sys.modules.update(mods)
    try:
        ar = {"_py2div": _py2div}
        exec(py2_compile(read("graphy/nodes/ar.py"), "graphy/nodes/ar.py"), ar)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    return ar, Nconv


# --------------------------------------------------------------------------
# cases
# --------------------------------------------------------------------------
from tests.golden.cases import MULTICONV_CASES, case_inputs, checksum  # noqa: E402


def run_tf_multiconv(tf, layers, hid, heads, z, ctx, hidden_sizes, n_z):
    tf.store.clear()
    for i, l in enumerate(hid):
        for k in "Vgb":
            tf.store["amc/layer_%d/%s" % (i, k)] = l[k].astype(np.float64)
    for i, l in enumerate(heads):
        for k in "Vgb":
            tf.store["amc/layer_out_%d/%s" % (i, k)] = l[k].astype(np.float64)
    out = layers["ar_multiconv2d"]("amc", RT(z), RT(ctx), list(hidden_sizes), [n_z, n_z])
    return [np.asarray(o) for o in out]


def run_theano_multiconv(ar, hid, heads, z, ctx, hidden_sizes, n_z, nl):
    w = {}
    np.random.seed(0)
    op = ar["multiconv2d"]("p", n_z, list(hidden_sizes), [n_z, n_z], (3, 3), False, nl=nl, w=w)
    for i, l in enumerate(hid):
        w["p_%d_w" % i] = RT(l["w"]); w["p_%d_s" % i] = RT(l["s"]); w["p_%d_b" % i] = RT(l["b"])
    for i, l in enumerate(heads):
        w["p_out_%d_w" % i] = RT(l["w"]); w["p_out_%d_s" % i] = RT(l["s"]); w["p_out_%d_b" % i] = RT(l["b"])
    out = op(RT(z), RT(ctx), w)
    return [np.asarray(o) for o in out]


def main():
    out_dir = HERE
    tf, layers, dist, train = load_tf_reference()
    ar, Nconv = load_theano_reference()

    # ---- masks (layers.py:115-141, ar.py:241-264) ---------------------------
    masks = {}
    for (n_in, n_out) in [(32, 64), (64, 64), (64, 32), (32, 160), (160, 160), (160, 32), (4, 8), (8, 4), (4, 4), (8, 8)]:
        for zd in (False, True):
            m = np.asarray(layers["get_conv_ar_mask"](3, 3, n_in, n_out, zd))
            masks["tf_%d_%d_%d" % (n_in, n_out, zd)] = np.packbits(m.astype(np.uint8).reshape(-1))
            masks["tf_%d_%d_%d_nnz" % (n_in, n_out, zd)] = np.int64(m.sum())
            lin = np.asarray(layers["get_linear_ar_mask"](n_in, n_out, zd))
            masks["lin_%d_%d_%d" % (n_in, n_out, zd)] = np.packbits(lin.astype(np.uint8).reshape(-1))
    # the Theano mask is built inline inside ar.conv2d and only visible through postup():
    # postup multiplies the update by the mask, so feeding all-ones recovers it (ar.py:369-373).
    for (n_in, n_out) in [(32, 64), (64, 32), (4, 8), (8, 4), (4, 4)]:
        for zd in (False, True):
            w = {}
            c = ar["conv2d"]("m", n_in, n_out, (3, 3), zd, False, w=w)
            m = _theano_mask_via_postup(c, w)
            masks["th_%d_%d_%d" % (n_in, n_out, zd)] = np.packbits(m.astype(np.uint8).reshape(-1))
            masks["th_%d_%d_%d_nnz" % (n_in, n_out, zd)] = np.int64(m.sum())
    np.savez_compressed(os.path.join(out_dir, "masks.npz"), **masks)

    # ---- multiconv (ar_multiconv2d / multiconv2d) ------------------------------
    mc = {}
    for ci, (name, variant, B, n_z, hidden, H, W, nl) in enumerate(MULTICONV_CASES):
        hid, heads, z, ctx = case_inputs(variant, B, n_z, hidden, H, W, seed=ci)
        if variant == "tf":
            m, s = run_tf_multiconv(tf, layers, hid, heads, z, ctx, hidden, n_z)
        else:
            m, s = run_theano_multiconv(ar, hid, heads, z, ctx, hidden, n_z, nl)
        mc[name + "_m"] = m
        mc[name + "_s"] = s
        mc[name + "_insum"] = np.float64(checksum(z, ctx, *[v for l in hid + heads for v in l.values()]))
        print(name, variant, m.shape, float(np.abs(m).max()), float(np.abs(s).max()))
    np.savez_compressed(os.path.join(out_dir, "multiconv.npz"), **mc)

    # ---- pad2dwithchannel (conv.py:71-83) -------------------------------------------
    x = np.random.RandomState(5).randn(2, 3, 4, 5).astype(np.float32)
    np.savez_compressed(os.path.join(out_dir, "pad.npz"), x=x, y=np.asarray(Nconv.pad2dwithchannel(RT(x), (3, 3))))

    # ---- IAFLayer.down (tf_train.py:46-95) -------------------------------------------
    down = {}
    down_tc = {}   # a tensor-core-eligible shape (z 32, h 64, 8x8), kept in its own file
    for name, kl_min, dims in (("kl0", 0.0, (4, 4, 8, 6, 6)), ("kl01", 0.1, (4, 4, 8, 6, 6)), ("kl5", 5.0, (4, 4, 8, 6, 6)),
                               ("tc_kl01", 0.1, (4, 32, 64, 8, 8)), ("tc_kl0", 0.0, (3, 32, 64, 8, 8))):
        B, zs, hs, H, W = dims
        rng = np.random.RandomState(11)
        hps = types.SimpleNamespace(h_size=hs, z_size=zs, kl_min=kl_min, batch_size=B, k=1)
        layer = train["IAFLayer"](hps, "train", False)
        f32 = lambda a: a.astype(np.float32).astype(np.float64)
        inp = f32(rng.randn(B, hs, H, W))
        layer.qz_mean = RT(f32(0.3 * rng.randn(B, zs, H, W)))
        layer.qz_logsd = RT(f32(0.2 * rng.randn(B, zs, H, W)))
        layer.up_context = RT(f32(0.1 * rng.randn(B, hs, H, W)))
        eps = f32(rng.randn(B, zs, H, W))
        hid, heads = O.make_params("tf", zs, [hs, hs], [zs, zs], seed=77)
        tf.store.clear()
        for i, l in enumerate(hid):
            for k in "Vgb":
                tf.store["ar_multiconv2d/layer_%d/%s" % (i, k)] = l[k].astype(np.float64)
        for i, l in enumerate(heads):
            for k in "Vgb":
                tf.store["ar_multiconv2d/layer_out_%d/%s" % (i, k)] = l[k].astype(np.float64)
        c1 = dict(V=f32(0.05 * rng.randn(3, 3, hs, 4 * zs + 2 * hs)), g=f32(rng.uniform(-.5, .5, 4 * zs + 2 * hs)),
                  b=f32(0.1 * rng.randn(4 * zs + 2 * hs)))
        c2 = dict(V=f32(0.05 * rng.randn(3, 3, zs + hs, hs)), g=f32(rng.uniform(-.5, .5, hs)), b=f32(0.1 * rng.randn(hs)))
        for k in "Vgb":
            tf.store["down_conv1/" + k] = c1[k]
            tf.store["down_conv2/" + k] = c2[k]
        # posterior.sample draws first, prior.sample second (tf_train.py:56-57 construct prior first)
        tf.noise[:] = [f32(rng.randn(B, zs, H, W)), eps]
        rec = {}
        orig = train["ar_multiconv2d"]

        def spy(nm, z, context, n_h, n_out, **kw):
            rec["z0"], rec["context"] = np.asarray(z).copy(), np.asarray(context).copy()
            o = orig(nm, z, context, n_h, n_out, **kw)
            rec["m"], rec["s"] = np.asarray(o[0]).copy(), np.asarray(o[1]).copy()
            return o
        train["ar_multiconv2d"] = spy
        try:
            output, kl_obj, kl_cost = layer.down(RT(inp))
        finally:
            train["ar_multiconv2d"] = orig
        # the six tensors IAFLayer.down slices out of down_conv1 (tf_train.py:53-54), re-derived
        x1 = layers["conv2d"]("down_conv1", tf.nn.elu(RT(inp)), 4 * zs + 2 * hs)
        pz_mean, pz_logsd, rz_mean, rz_logsd, down_context, h_det = [np.asarray(t) for t in
                                                                     train["split"](x1, 1, [zs] * 4 + [hs] * 2)]
        (down_tc if name.startswith("tc_") else down).update({name + "_" + k: v for k, v in dict(
            inp=inp, qz_mean=np.asarray(layer.qz_mean), qz_logsd=np.asarray(layer.qz_logsd),
            up_context=np.asarray(layer.up_context), eps=eps, pz_mean=pz_mean, pz_logsd=pz_logsd,
            rz_mean=rz_mean, rz_logsd=rz_logsd, down_context=down_context, z0=rec["z0"], context=rec["context"],
            m=rec["m"], s=rec["s"], output=np.asarray(output), kl_obj=np.asarray(kl_obj),
            kl_cost=np.asarray(kl_cost), kl_min=np.float64(kl_min)).items()})
    np.savez_compressed(os.path.join(out_dir, "iaflayer_down.npz"), **down)
    # the tensor-core shape keeps only what its test reads (inp, context and output would take the file past 1 MB)
    np.savez_compressed(os.path.join(out_dir, "iaflayer_down_tc.npz"), **{k: (v.astype(np.float32) if getattr(v, "ndim", 0) else v)
                                                                         for k, v in down_tc.items()
                                                                         if k.split("_", 2)[2] not in ("inp", "context", "output")})

    # ---- distributions.py (logsumexp / compute_lowerbound / repeat / logps) -----------
    rng = np.random.RandomState(3)
    a = rng.randn(6, 4)
    b = rng.randn(6, 4)
    d = dict(a=a, b=b,
             logsumexp=np.asarray(dist["logsumexp"](RT(a))),
             lb_k4=np.asarray(dist["compute_lowerbound"](RT(a.reshape(-1)), RT(b.reshape(-1)), 4)),
             lb_k1=np.asarray(dist["compute_lowerbound"](RT(a.reshape(-1)), RT(b.reshape(-1)), 1)),
             repeat3=np.asarray(dist["repeat"](RT(a), 3)),
             logps=np.asarray(dist["gaussian_diag_logps"](RT(a), RT(0.3 * b), RT(b))))
    np.savez_compressed(os.path.join(out_dir, "distributions.npz"), **d)
    print("golden fixtures written to", out_dir)


def _theano_mask_via_postup(conv, w):
    """ar.py:369-373: updates[w[name_w+'_w']] = mask * updates[...].  Theano keys the updates
    dict by the shared variable; the stand-in keys by object id."""
    key = w["m_w"]

    class ById(dict):
        def __getitem__(self, k):
            return dict.__getitem__(self, id(k))

        def __setitem__(self, k, v):
            dict.__setitem__(self, id(k), v)
    upd = ById()
    upd[key] = RT(np.ones(key.shape))
    upd = conv.postup(upd, w)
    return np.asarray(upd[key])


if __name__ == "__main__":
    main()
