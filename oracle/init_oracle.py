"""CPU oracle of the data-dependent initialisation pass of the masked-AR stack (TEST INFRASTRUCTURE ONLY).

A numpy restatement, in the dtype of the inputs (float64 for the truth oracle), of the branches both reference
front-ends take once before the first training step: TF ``conv2d(..., init=True)`` reached through ``ar_conv2d``
(tf_utils/layers.py:38-51, 145-154; built by tf_train.py:226-228) and Theano ``ar.conv2d`` with ``w['__init']``
(graphy/nodes/ar.py:331-353; set by models.py:541-544).  Same status as oracle/iaf_oracle.py: only tests may import
it; the fixture tests/golden/data_init.npz is produced by executing the reference's own lines
(tests/golden/make_golden_init.py).
"""
import numpy as np

from oracle.iaf_oracle import (get_conv_ar_mask, nonlinearity, tf_effective_weight, theano_ar_conv2d,
                               xcorr2d_same)


def _tf_layer(x, layer, zd):
    """layers.py:38-51 (init_scale = 1): x_init = xcorr(x, l2_normalize(mask*V)); scale = 1/sqrt(var + 1e-10);
    g = log(scale)/3; b = -mean*scale; returns scale*(x_init - mean)."""
    V = layer["V"]
    mask = get_conv_ar_mask(V.shape[0], V.shape[1], V.shape[2], V.shape[3], zd)
    xi = xcorr2d_same(x, tf_effective_weight(V, np.zeros(V.shape[3], V.dtype), mask))  # exp(0) * l2_normalize
    m, v = xi.mean(axis=(0, 2, 3)), xi.var(axis=(0, 2, 3))
    scale = 1.0 / np.sqrt(v + 1e-10)
    return scale.reshape(1, -1, 1, 1) * (xi - m.reshape(1, -1, 1, 1)), (np.log(scale) / 3.0, -m * scale), 0


def _theano_layer(x, layer, zd):
    """ar.py:304-353: h = the layer's forward with the CURRENT s, b; any std == 0 -> skipped (parameters unchanged,
    h returned); else s = -log(std)/3, h /= std, b = -mean(h), h -= mean(h)."""
    h = theano_ar_conv2d(x, layer, zd)
    std = h.std(axis=(0, 2, 3))
    nzero = int((std == 0).sum())
    if nzero:
        return h, (layer["s"], layer["b"]), nzero
    h = h / std.reshape(1, -1, 1, 1)
    mean = h.mean(axis=(0, 2, 3))
    return h - mean.reshape(1, -1, 1, 1), (-np.log(std) / 3.0, -mean), 0


def data_init(variant, z, context, hidden, heads, nl="elu"):
    """The init pass of the stack, layer by layer: each layer's returned tensor feeds the next, the context is added
    after hidden layer 0 and nl follows every hidden layer (layers.py:161-166 / ar.py:400-409).  Statistics are per
    output channel over (batch, H, W) with population variance (tf.nn.moments; Theano std, ddof 0).
    hidden/heads: layer dicts as in oracle.iaf_oracle (tf: V, g, b -- g and b are not read; theano: w, s, b).
    Returns (head outputs, [(new g|s, new b)] per layer with hidden layers first, [zero-std channel count] per layer:
    Theano skipped the layers where it is > 0, TF always 0)."""
    one = _tf_layer if variant == "tf" else _theano_layer
    f = nonlinearity(nl)
    params, zeros, x = [], [], z
    for i, layer in enumerate(hidden):
        x, p, n = one(x, layer, False)
        params.append(p)
        zeros.append(n)
        if i == 0:
            x = x + context
        x = f(x)
    outs = []
    for layer in heads:
        o, p, n = one(x, layer, True)
        outs.append(o)
        params.append(p)
        zeros.append(n)
    return outs, params, zeros
