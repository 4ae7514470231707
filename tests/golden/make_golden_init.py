#!/usr/bin/env python
"""Golden vectors of the data-dependent initialisation pass, produced by EXECUTING the reference's own source:
``ar_multiconv2d`` (tf_utils/layers.py:158-166) under ``arg_scope([conv2d], init=True)``, which reaches every AR conv
through ``ar_conv2d`` (145-154) and takes the init branch of ``conv2d`` (38-51), and ``multiconv2d``
(graphy/nodes/ar.py:378-416) called with ``w['__init']`` set (331-353), as tf_train.py:226-228 and
models.py:541-544 do once before training.

Run in the build container only (needs /root/reference):  python tests/golden/make_golden_init.py
Writes tests/golden/data_init.npz.  Same approach as make_golden.py (python2 -> python3 syntax shims, eager ndarray
stand-ins, cuDNN replaced by torch CPU float64 convolution), plus what the init branches call on top of the forward:
tf.contrib's arg_scope / add_arg_scope (nested scopes merge their keyword arguments), tf.nn.moments, tf.sqrt,
get_variable creating a variable from its initializer, and Theano's set_value.  Inputs are float32 values; the pass runs
in float64; the fixture holds the inputs and what the reference returned and stored.
"""
import contextlib
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
from oracle import iaf_oracle as O  # noqa: E402  (only for make_params / make_inputs seeds)
from tests.golden import make_golden as MG  # noqa: E402

RT = MG.RT

INIT_CASES = [
    # name, variant, B, n_z, hidden, H, W, nl
    ("tf_8_8", "tf", 3, 4, [8, 8], 5, 7, "elu"),       # ragged H != W
    ("tf_zero_col", "tf", 2, 4, [8], 4, 5, "elu"),     # one all-zero V column: the 1e5 branch
    ("th_8", "theano", 3, 4, [8], 5, 6, "elu"),        # starting from non-zero s, b
    ("th_skip", "theano", 2, 4, [8], 4, 4, "elu"),     # a constant head channel: that conv is skipped
    ("th_depth0", "theano", 2, 4, [], 5, 5, "elu"),    # depth_ar = 0
    ("tf_tc", "tf", 2, 16, [32], 8, 8, "elu"),         # tensor-core-eligible shape
]


def case_data(ci):
    """Seeded float32 inputs of case ci in the reference layouts, with the case's special entries applied."""
    name, variant, B, n_z, hidden, H, W, nl = INIT_CASES[ci]
    hid, heads = O.make_params(variant, n_z, hidden, [n_z, n_z], seed=200 + ci)
    z, ctx = O.make_inputs(B, n_z, hidden[0] if hidden else n_z, H, W, seed=300 + ci)
    if name == "tf_zero_col":
        hid[0]["V"][..., 3] = 0.0
    if name == "th_skip":
        heads[1]["w"][2] = 0.0  # output channel 2 of head 1 is the constant b[2]
    return hid, heads, z, ctx


# --------------------------------------------------------------------------
# TF: layers.py with a merging arg_scope and the init-branch primitives
# --------------------------------------------------------------------------
def load_tf_init_reference():
    tf = MG.TFShim()
    stack = [{}]

    @contextlib.contextmanager
    def arg_scope(fns, **kw):  # tf.contrib: a nested scope starts from a copy of the enclosing one and updates it
        cur = {k: dict(v) for k, v in stack[-1].items()}
        for f in fns:
            cur.setdefault(getattr(f, "_scope_key", f.__name__), {}).update(kw)
        stack.append(cur)
        try:
            yield
        finally:
            stack.pop()

    def add_arg_scope(f):
        def g(*a, **k):
            kk = dict(stack[-1].get(f.__name__, {}))
            kk.update(k)
            return f(*a, **kk)
        g._scope_key = f.__name__
        g.__name__ = f.__name__
        return g

    def moments(x, axes):
        x = np.asarray(x)
        return RT(x.mean(axis=tuple(axes))), RT(x.var(axis=tuple(axes)))

    tf.nn.moments = moments
    tf.sqrt = lambda x: RT(np.sqrt(np.asarray(x)))
    tf.random_normal_initializer = lambda *a, **k: None  # V is always present in the store
    get_existing = tf.get_variable

    def get_variable(name, shape=None, dtype=None, initializer=None):
        key = "/".join(tf.scope + [name])
        if key not in tf.store:
            tf.store[key] = np.asarray(initializer, dtype=np.float64)
        return get_existing(name, shape, dtype)
    tf.get_variable = get_variable

    fw = types.ModuleType("tensorflow.contrib.framework.python.ops")
    fw.arg_scope, fw.add_arg_scope = arg_scope, add_arg_scope
    mods = {"tensorflow": tf, "tensorflow.contrib": types.ModuleType("c"),
            "tensorflow.contrib.framework": types.ModuleType("c"),
            "tensorflow.contrib.framework.python": types.ModuleType("c"),
            "tensorflow.contrib.framework.python.ops": fw}
    saved = {k: sys.modules.get(k) for k in mods}
    sys.modules.update(mods)
    try:
        layers = {"_py2div": MG._py2div}
        exec(MG.py2_compile(MG.read("tf_utils/layers.py"), "tf_utils/layers.py"), layers)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    return tf, layers, arg_scope


def run_tf(tf, layers, arg_scope, hid, heads, z, ctx, hidden_sizes, n_z):
    tf.store.clear()  # only V exists before the init pass: g and b are created by it
    for i, l in enumerate(hid):
        tf.store["amc/layer_%d/V" % i] = l["V"].astype(np.float64)
    for i, l in enumerate(heads):
        tf.store["amc/layer_out_%d/V" % i] = l["V"].astype(np.float64)
    with arg_scope([layers["conv2d"]], init=True):
        out = layers["ar_multiconv2d"]("amc", RT(z), RT(ctx), list(hidden_sizes), [n_z, n_z])
    scopes = ["layer_%d" % i for i in range(len(hid))] + ["layer_out_%d" % i for i in range(len(heads))]
    params = [(np.asarray(tf.store["amc/%s/g" % s]), np.asarray(tf.store["amc/%s/b" % s])) for s in scopes]
    return [np.asarray(o) for o in out], params


# --------------------------------------------------------------------------
# Theano: ar.py with w['__init'] and set_value
# --------------------------------------------------------------------------
def _set_value(self, v):  # Theano shared variable: overwrite in place
    self[...] = np.asarray(v)


def run_theano(ar, hid, heads, z, ctx, hidden_sizes, n_z, nl):
    w = {}
    np.random.seed(0)
    op = ar["multiconv2d"]("p", n_z, list(hidden_sizes), [n_z, n_z], (3, 3), False, nl=nl, w=w)
    names = ["p_%d" % i for i in range(len(hid))] + ["p_out_%d" % i for i in range(len(heads))]
    for nm, l in zip(names, hid + heads):
        w[nm + "_w"], w[nm + "_s"], w[nm + "_b"] = RT(l["w"]), RT(l["s"]), RT(l["b"])
    w["__init"] = RT(np.zeros(()))
    out = op(RT(z), RT(ctx), w)
    params = [(np.asarray(w[nm + "_s"]).copy(), np.asarray(w[nm + "_b"]).copy()) for nm in names]
    return [np.asarray(o) for o in out], params


def main():
    tf, layers, arg_scope = load_tf_init_reference()
    ar, _ = MG.load_theano_reference()
    RT.set_value = _set_value
    g = {}
    for ci, (name, variant, B, n_z, hidden, H, W, nl) in enumerate(INIT_CASES):
        hid, heads, z, ctx = case_data(ci)
        if variant == "tf":
            outs, params = run_tf(tf, layers, arg_scope, hid, heads, z, ctx, hidden, n_z)
        else:
            outs, params = run_theano(ar, hid, heads, z, ctx, hidden, n_z, nl)
        keys = ("V", "g", "b") if variant == "tf" else ("w", "s", "b")
        for i, l in enumerate(hid + heads):
            for k in keys:
                g["%s/in/%d/%s" % (name, i, k)] = l[k]
        g[name + "/z"], g[name + "/ctx"] = z, ctx
        for k, o in enumerate(outs):
            g["%s/out/%d" % (name, k)] = o
        for i, (s, b) in enumerate(params):
            g["%s/scale/%d" % (name, i)], g["%s/bias/%d" % (name, i)] = s, b
        print(name, variant, [o.shape for o in outs], float(np.abs(outs[0]).max()))
    np.savez_compressed(os.path.join(HERE, "data_init.npz"), **g)
    print("written", os.path.join(HERE, "data_init.npz"), len(g), "arrays")


if __name__ == "__main__":
    main()
