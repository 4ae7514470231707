"""Host side of the B200 IAF step: the reference's python operator signatures over the C ABI.

PyTorch tensors are used as device storage and for the current stream only; all compute
is in libiaf_b200.so (include/iaf_b200.h).  Three entry points mirror the reference:

* ``ar_multiconv2d(name, x, context, n_h, n_out, nl, params=...)``
      tf_utils/layers.py:158-166 (called at tf_train.py:69)
* ``multiconv2d(name, n_in, n_h, n_out, size_kernel, flipmask, nl, w)`` -> callable
      graphy/nodes/ar.py:378-423 (called at models.py:92,170,281)
* ``iaf_step(z, context, ...)`` -- the fused superset: the stack plus the caller's
      ``arw_mean*=.1; arw_logsd*=.1; z=(z-arw_mean)/exp(arw_logsd); logqs+=arw_logsd``
      (models.py:282-285, tf_train.py:70-72)

Both reference functions are graph builders called once; here they run eagerly per batch,
so the masked / normalised / packed weights are cached on the operator and re-packed only
when a parameter tensor changes (SURVEY F9).
"""
import ctypes as C
import os
import warnings

import numpy as np
import torch

from . import _lib
from .masks import theano_conv_ar_mask


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _stream(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _check_input(t, name, shape=None):
    if not isinstance(t, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor" % name)
    if not t.is_cuda:
        raise RuntimeError("iaf_b200: %s is on %s; this operator only runs on CUDA (no CPU fallback)" % (name, t.device))
    if t.dtype != torch.float32:
        raise TypeError("%s must be float32 (reference floatX / tf.float32), got %s" % (name, t.dtype))
    if shape is not None and tuple(t.shape) != tuple(shape):
        raise ValueError("%s has shape %s, expected %s" % (name, tuple(t.shape), tuple(shape)))
    return t.contiguous()


class IAFOperator(object):
    """One masked-AR conv stack (+ fused affine update) bound to raw reference parameters.

    variant: "tf" (tf_utils/layers.py numerics) or "theano" (graphy/nodes/ar.py numerics).
    layers:  list of (w, scale, bias) tensors, hidden layers first then heads, in the
             reference's layouts: tf V [3,3,Cin,Cout], g, b; theano w [Cout,Cin+1,3,3], s, b.
    """

    def __init__(self, variant, n_z, hidden, heads, nl="elu", path="auto", checknan=None):
        """checknan="raise": the reference driver's NaN guard (graphy/function.py:107-110 raises "NaN detected" when the sum
        of a minibatch's outputs is NaN; train.py:211, tf_train.py:283-285 stop likewise): after a step, the per-sample
        logdet (a sum over every element the kernel produced) is checked on the host.  Off by default: it synchronises."""
        if checknan not in (None, "raise"):
            raise ValueError("checknan must be None or 'raise'")
        self.checknan = checknan
        if variant not in _lib.VARIANTS:
            raise ValueError("variant must be 'tf' or 'theano'")
        if nl not in _lib.NLS:
            raise NotImplementedError("nonlinearity %r is not available in the fused kernel" % (nl,))
        if path not in _lib.PATHS:
            raise ValueError("path must be one of %s" % sorted(_lib.PATHS))
        hidden, heads = [int(h) for h in hidden], [int(h) for h in heads]
        if len(hidden) > _lib.IAF_MAX_HIDDEN:
            raise NotImplementedError("at most %d hidden layers" % _lib.IAF_MAX_HIDDEN)
        if not 1 <= len(heads) <= _lib.IAF_MAX_HEADS:
            raise NotImplementedError("n_out must have 1 or 2 entries")
        self.variant, self.n_z, self.hidden, self.heads, self.nl, self.path = variant, int(n_z), hidden, heads, nl, path
        self._layers = None
        self._epoch = 0       # bumped by set_weights()/invalidate(): part of the packed-weights cache key
        self._plans = {}      # (H, W, device index) -> [handle, packed_key]
        self._lib = _lib.lib()

    # ---- parameters ---------------------------------------------------------------
    def set_weights(self, layers):
        n = len(self.hidden) + len(self.heads)
        if len(layers) != n:
            raise ValueError("expected %d (w, scale, bias) triples, got %d" % (n, len(layers)))
        sizes = [self.n_z] + self.hidden
        out = []
        for i, (w, s, b) in enumerate(layers):
            cin = sizes[min(i, len(self.hidden))]
            cout = self.hidden[i] if i < len(self.hidden) else self.heads[i - len(self.hidden)]
            wshape = (3, 3, cin, cout) if self.variant == "tf" else (cout, cin + 1, 3, 3)
            out.append((_check_input(w, "w[%d]" % i, wshape), _check_input(s, "scale[%d]" % i, (cout,)),
                        _check_input(b, "bias[%d]" % i, (cout,))))
        same = self._layers is not None and len(self._layers) == len(out) and all(
            a is b for la, lb in zip(self._layers, out) for a, b in zip(la, lb))
        self._layers = out
        if not same:
            self._epoch += 1  # different tensor objects: never reuse a packed copy across a re-binding
        return self

    def _weights_key(self, layers=None):
        """Identity of the packed weights: (storage, version counter) of every parameter tensor plus the operator's own
        epoch.  In-place updates through ``.data`` (``p.data.copy_``, the usual spelling in older training loops and in
        ports of the reference's ``postup``) do NOT bump ``_version``; callers that update parameters that way call
        ``invalidate()`` (or ``set_weights`` with new tensors, which does).  Calls recorded for autograd never trust the
        packed copy: they invalidate first (two small launches per call), see ``_for_training``."""
        ls = self._layers if layers is None else layers
        return (self._epoch,) + tuple((t.data_ptr(), t._version) for l in ls for t in l)

    def invalidate(self):
        """Forget the packed weights: the next call re-runs iaf_pack_weights from the raw parameter tensors."""
        self._epoch += 1
        return self

    def _needs_grad(self, *tensors):
        if not torch.is_grad_enabled():
            return False
        ts = [t for t in tensors if t is not None] + [t for l in (self._layers or []) for t in l]
        return any(t.requires_grad for t in ts)

    # ---- plans ----------------------------------------------------------------------
    def _plan(self, H, W, device, layers=None, pack=True):
        """Plan for (H, W, device) with the packed weights of ``layers`` (default: the current set_weights());
        ``pack=False``: the plan as it is (data_init packs for itself)."""
        key = (H, W, device.index)
        ent = self._plans.get(key)
        if ent is None:
            d = _lib.IafDesc()
            d.variant = _lib.VARIANTS[self.variant]
            d.n_z = self.n_z
            d.n_hidden = len(self.hidden)
            for i, h in enumerate(self.hidden):
                d.hidden[i] = h
            d.n_heads = len(self.heads)
            for i, h in enumerate(self.heads):
                d.head[i] = h
            d.H, d.W = H, W
            d.nl = _lib.NLS[self.nl]
            d.path = _lib.PATHS[self.path]
            handle = C.c_void_p()
            with torch.cuda.device(device):
                _lib.check(self._lib.iaf_plan_create(C.byref(handle), C.byref(d)))
            ent = [handle, None]
            self._plans[key] = ent
        if not pack:
            return ent[0]
        if layers is None:
            layers = self._layers
        if layers is None:
            raise RuntimeError("IAFOperator.set_weights() has not been called")
        wk = self._weights_key(layers)
        if ent[1] != wk:
            n = len(layers)
            arr = lambda j: (C.c_void_p * n)(*[l[j].data_ptr() for l in layers])
            with torch.cuda.device(device):
                _lib.check(self._lib.iaf_pack_weights(ent[0], arr(0), arr(1), arr(2), _stream(device)))
            ent[1] = wk
        return ent[0]

    def __del__(self):
        try:
            for ent in self._plans.values():
                self._lib.iaf_plan_destroy(ent[0])
        except Exception:
            pass

    # ---- introspection --------------------------------------------------------------
    def path_used(self, H, W, device, entry=None):
        """Kernel family this operator runs on for (H, W): "tc" or "simt".  With ``entry`` ("step" | "multiconv" |
        "layer") the answer is for THAT entry point: an ``path="auto"`` operator may serve one entry on the SIMT kernel
        although the plan is a tensor-core plan (e.g. ``layer`` when its scratch does not fit); ``path="tc"`` operators
        raise NotImplementedError from such a call instead of slowing down 10-40x."""
        plan = self._plan(H, W, torch.device(device))
        if entry is None:
            return _lib.PATH_NAMES[self._lib.iaf_plan_path(plan)]
        rc = self._lib.iaf_plan_path_for_entry(plan, _lib.ENTRIES[entry])
        if rc < 0:
            _lib.check(rc)
        return _lib.PATH_NAMES[rc]

    def backward_path(self, H, W, device):
        """Kernels behind the backward entries for (H, W): "simt" (exact fp32), "tc-dgrad" (data gradient on the tensor
        cores) or "tc" (data and weight gradient on the tensor cores)."""
        rc = self._lib.iaf_plan_bwd_path(self._plan(H, W, torch.device(device)))
        if rc < 0:
            _lib.check(rc)
        return ("simt", "tc-dgrad", "tc")[rc]

    def launch_count(self):
        return sum(int(self._lib.iaf_plan_launch_count(e[0])) for e in self._plans.values())

    def algorithmic_bytes(self, B, H, W, device):
        return int(self._lib.iaf_plan_algorithmic_bytes(self._plan(H, W, torch.device(device)), B))

    def algorithmic_flops(self, B, H, W, device):
        return float(self._lib.iaf_plan_algorithmic_flops(self._plan(H, W, torch.device(device)), B))

    # ---- calls ----------------------------------------------------------------------
    def _shapes(self, z, context):
        z = _check_input(z, "z")
        if z.dim() != 4 or z.shape[1] != self.n_z:
            raise ValueError("z must be [B,%d,H,W], got %s" % (self.n_z, tuple(z.shape)))
        B, _, H, W = z.shape
        if self.hidden:
            context = _check_input(context, "context", (B, self.hidden[0], H, W))
            if context.device != z.device:
                raise ValueError("z and context are on different devices")
        else:
            context = None  # never added when there is no hidden layer (ar.py:399-403, SURVEY F8)
        return z, context, B, H, W

    def multiconv(self, z, context):
        """The un-fused stack: list of head outputs (ar.py:396-416 / layers.py:158-166).  Differentiable: when an
        input or a parameter requires grad the call is recorded for autograd (backward = iaf_multiconv_bwd)."""
        if self._needs_grad(z, context):
            self.invalidate()  # training: parameters may have been stepped through .data since the last call
            flat = [t for l in self._layers for t in l]
            return list(_MulticonvFn.apply(self, z, context if self.hidden else None, *flat))
        return self._multiconv_raw(z, context)

    def _multiconv_raw(self, z, context):
        z, context, B, H, W = self._shapes(z, context)
        plan = self._plan(H, W, z.device)
        outs = [torch.empty((B, h, H, W), device=z.device, dtype=torch.float32) for h in self.heads]
        arr = (C.c_void_p * len(outs))(*[o.data_ptr() for o in outs])
        with torch.cuda.device(z.device):
            _lib.check(self._lib.iaf_multiconv_fwd(plan, _ptr(z), _ptr(context), arr, B, _stream(z.device)))
        return outs

    def step(self, z, context, want_logsd=True, want_logdet=True):
        """(z', arw_logsd [B,C,H,W], logdet [B]); logqs_new = logqs + arw_logsd.  Differentiable: when an input or a
        parameter requires grad the call is recorded for autograd (backward = iaf_step_bwd, SURVEY 8f-4)."""
        if self._needs_grad(z, context):
            self.invalidate()  # training: parameters may have been stepped through .data since the last call
            flat = [t for l in self._layers for t in l]
            z_out, logsd, logdet = _StepFn.apply(self, z, context if self.hidden else None, *flat)
            self._nan_guard(logdet)
            return z_out, (logsd if want_logsd else None), (logdet if want_logdet else None)
        out = self._step_raw(z, context, want_logsd, want_logdet or self.checknan == "raise")
        self._nan_guard(out[2])
        return out[0], out[1], (out[2] if want_logdet else None)

    def data_init(self, z, context, names=None):
        """Data-dependent initialisation on one batch (iaf_multiconv_init): the pass the reference runs once before
        training -- TF ``init=True`` (layers.py:38-51), Theano ``w['__init']`` (ar.py:331-353).  Writes the new g|s and
        b into the bound parameter tensors in place (``copy_``), so the next call re-packs; returns the pass's head
        outputs.  Theano layers with a zero-std channel keep their parameters and warn with the reference's text;
        ``names`` (one per layer, hidden layers first) are the layer names that text uses."""
        if self._layers is None:
            raise RuntimeError("IAFOperator.set_weights() has not been called")
        n = len(self._layers)
        if names is None:
            names = ["layer_%d" % i for i in range(len(self.hidden))] + ["layer_out_%d" % k for k in range(len(self.heads))]
        with torch.no_grad():
            z, context, B, H, W = self._shapes(z, context)
            dev = z.device
            plan = self._plan(H, W, dev, pack=False)
            new_s = [torch.empty_like(l[1]) for l in self._layers]
            new_b = [torch.empty_like(l[2]) for l in self._layers]
            outs = [torch.empty((B, h, H, W), device=dev, dtype=torch.float32) for h in self.heads]
            skipped = torch.zeros((n,), device=dev, dtype=torch.int32)
            arr = lambda ts: (C.c_void_p * n)(*[t.data_ptr() for t in ts])
            cur = (arr([l[1] for l in self._layers]), arr([l[2] for l in self._layers])) if self.variant == "theano" \
                else (None, None)  # TF: the init branch does not read g, b
            self._plans[(H, W, dev.index)][1] = None  # the init pass uses the packed buffers as scratch
            with torch.cuda.device(dev):
                _lib.check(self._lib.iaf_multiconv_init(plan, _ptr(z), _ptr(context), arr([l[0] for l in self._layers]),
                                                        cur[0], cur[1], arr(new_s), arr(new_b),
                                                        (C.c_void_p * len(outs))(*[o.data_ptr() for o in outs]),
                                                        _ptr(skipped), B, _stream(dev)))
            for l, s, b in zip(self._layers, new_s, new_b):
                l[1].copy_(s)  # bumps _version: every plan of this operator re-packs on its next call
                l[2].copy_(b)
            for name, nzero in zip(names, skipped.tolist()):
                if nzero > 0:  # ar.py:336
                    warnings.warn("Stdev=0 for %d features in %s. Skipping data-dependent init." % (nzero, name),
                                  RuntimeWarning)
        return outs

    def _nan_guard(self, logdet):
        if self.checknan == "raise" and bool(torch.isnan(logdet.detach().sum())):
            raise FloatingPointError("NaN detected")  # graphy/function.py:110

    def _step_raw(self, z, context, want_logsd=True, want_logdet=True):
        z, context, B, H, W = self._shapes(z, context)
        plan = self._plan(H, W, z.device)
        z_out = torch.empty_like(z)
        logsd = torch.empty_like(z) if want_logsd else None
        logdet = torch.empty((B,), device=z.device, dtype=torch.float32) if want_logdet else None
        with torch.cuda.device(z.device):
            _lib.check(self._lib.iaf_step_fwd(plan, _ptr(z), _ptr(context), _ptr(z_out), _ptr(logsd), _ptr(logdet),
                                              B, _stream(z.device)))
        return z_out, logsd, logdet

    def _multiconv_train_raw(self, z, context):
        """iaf_multiconv_fwd_train: the un-fused stack plus the hidden activations its backward needs."""
        z, context, B, H, W = self._shapes(z, context)
        plan = self._plan(H, W, z.device)
        outs = [torch.empty((B, h, H, W), device=z.device, dtype=torch.float32) for h in self.heads]
        hidden = [torch.empty((B, h, H, W), device=z.device, dtype=torch.float32) for h in self.hidden]
        oarr = (C.c_void_p * len(outs))(*[o.data_ptr() for o in outs])
        harr = (C.c_void_p * max(1, len(hidden)))(*[h.data_ptr() for h in hidden])
        with torch.cuda.device(z.device):
            _lib.check(self._lib.iaf_multiconv_fwd_train(plan, _ptr(z), _ptr(context), oarr, harr, B, _stream(z.device)))
        return outs, hidden

    def _step_train_raw(self, z, context):
        """iaf_step_fwd_train: the step plus the hidden activations the backward needs (kept by the same kernels)."""
        z, context, B, H, W = self._shapes(z, context)
        plan = self._plan(H, W, z.device)
        z_out, logsd = torch.empty_like(z), torch.empty_like(z)
        logdet = torch.empty((B,), device=z.device, dtype=torch.float32)
        hidden = [torch.empty((B, h, H, W), device=z.device, dtype=torch.float32) for h in self.hidden]
        harr = (C.c_void_p * max(1, len(hidden)))(*[h.data_ptr() for h in hidden])
        with torch.cuda.device(z.device):
            _lib.check(self._lib.iaf_step_fwd_train(plan, _ptr(z), _ptr(context), _ptr(z_out), _ptr(logsd), _ptr(logdet),
                                                    harr, B, _stream(z.device)))
        return z_out, logsd, logdet, hidden

    def step_host(self, z, context, z_out, logsd_out, logdet_out):
        """End-to-end entry on HOST tensors (pinned or pageable): H2D, step, D2H, sync."""
        for t in (z, context, z_out, logsd_out, logdet_out):
            if t is not None and (t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous()):
                raise ValueError("step_host takes contiguous float32 CPU tensors")
        B, _, H, W = z.shape
        device = torch.device("cuda", torch.cuda.current_device())
        plan = self._plan(H, W, device)
        _lib.check(self._lib.iaf_step_fwd_host(plan, _ptr(z), _ptr(context), _ptr(z_out), _ptr(logsd_out),
                                               _ptr(logdet_out), B, _stream(device)))
        return z_out, logsd_out, logdet_out

    def submit_host(self, z, context, z_out, logsd_out, logdet_out):
        """Pipelined host entry: enqueue H2D + step + D2H of one batch and return at once (pinned CPU tensors,
        valid until wait_host()).  Consecutive batches overlap copy-in, compute and copy-out."""
        for t in (z, context, z_out, logsd_out, logdet_out):
            if t is not None and (t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous() or not t.is_pinned()):
                raise ValueError("submit_host takes pinned contiguous float32 CPU tensors")
        B, _, H, W = z.shape
        device = torch.device("cuda", torch.cuda.current_device())
        self._host_plan = self._plan(H, W, device)
        # (weights packed on the caller's stream: the library orders its private compute stream after it, one event)
        _lib.check(self._lib.iaf_step_submit_host(self._host_plan, _ptr(z), _ptr(context), _ptr(z_out), _ptr(logsd_out),
                                                  _ptr(logdet_out), B))

    def wait_host(self):
        if getattr(self, "_host_plan", None) is not None:
            _lib.check(self._lib.iaf_host_wait(self._host_plan))

    def layer(self, eps, post_mean, post_logsd, prior_mean, prior_logsd, context, want_kl=True):
        """Fused posterior-sample -> IAF step -> KL block (tf_train.py:56-85, models.py:273-328).
        Returns (z', kl [B,C,H,W] or None, kl_bc [B,C], kl_cost [B]).  Differentiable: when an input or a parameter
        requires grad the call is ONE autograd node (backward = iaf_layer_bwd; confirmed on a B200 in round 2:
        worst relative gradient error 6.4e-4 on the whole training objective).  IAF_LAYER_AUTOGRAD=0 switches it off."""
        if os.environ.get("IAF_LAYER_AUTOGRAD", "1") != "0" and self._needs_grad(eps, post_mean, post_logsd, prior_mean,
                                                                                   prior_logsd, context):
            self.invalidate()  # training: parameters may have been stepped through .data since the last call
            flat = [t for l in self._layers for t in l]
            z_out, kl, kl_bc, kl_cost = _LayerFn.apply(self, eps, post_mean, post_logsd, prior_mean, prior_logsd,
                                                       context if self.hidden else None, *flat)
            return z_out, (kl if want_kl else None), kl_bc, kl_cost
        return self._layer_raw(eps, post_mean, post_logsd, prior_mean, prior_logsd, context, want_kl)

    def _layer_raw(self, eps, post_mean, post_logsd, prior_mean, prior_logsd, context, want_kl=True):
        eps, context, B, H, W = self._shapes(eps, context)
        ts = [_check_input(t, n, eps.shape) for t, n in ((post_mean, "post_mean"), (post_logsd, "post_logsd"),
                                                          (prior_mean, "prior_mean"), (prior_logsd, "prior_logsd"))]
        plan = self._plan(H, W, eps.device)
        z_out = torch.empty_like(eps)
        kl = torch.empty_like(eps) if want_kl else None
        kl_bc = torch.empty((B, self.n_z), device=eps.device, dtype=torch.float32)
        kl_cost = torch.empty((B,), device=eps.device, dtype=torch.float32)
        with torch.cuda.device(eps.device):
            _lib.check(self._lib.iaf_layer_fwd(plan, _ptr(eps), _ptr(ts[0]), _ptr(ts[1]), _ptr(ts[2]), _ptr(ts[3]),
                                               _ptr(context), _ptr(z_out), _ptr(kl), _ptr(kl_bc), _ptr(kl_cost), B,
                                               _stream(eps.device)))
        return z_out, kl, kl_bc, kl_cost

    # ---- backward (SURVEY 8f-4) -------------------------------------------------------
    def _backward(self, kind, z, context, layers, grads_out, need_params, saved=None):
        """Shared driver of iaf_step_bwd / iaf_step_bwd_saved / iaf_multiconv_bwd.  ``layers`` are the parameter
        tensors the forward used; ``saved`` = (z_out, logsd, [hidden]) kept by iaf_step_fwd_train (then ``context``
        is only a shape template for its gradient).  Returns (g_z, g_context or None, [g_w], [g_scale], [g_bias])
        (lists None when not needed)."""
        z, context, B, H, W = self._shapes(z, context)
        dev = z.device
        plan = self._plan(H, W, dev, layers)
        n = len(layers)
        arr = lambda ts: (C.c_void_p * n)(*[t.data_ptr() for t in ts])
        g_z = torch.empty_like(z)
        g_ctx = torch.empty_like(context) if context is not None else None
        gw = gs = gb = None
        if need_params:
            gw, gs, gb = ([torch.empty_like(l[j]) for l in layers] for j in range(3))
        pa = lambda ts: arr(ts) if ts is not None else None
        with torch.cuda.device(dev):
            if kind == "step":
                g_zout, g_logsd, g_logdet = grads_out
                if g_zout is None:
                    g_zout = torch.zeros_like(z)
                g_zout, g_logsd, g_logdet = (None if t is None else _check_input(t, "grad") for t in (g_zout, g_logsd, g_logdet))
                if saved is not None:
                    z_out, logsd, hidden = saved
                    harr = (C.c_void_p * max(1, len(hidden)))(*[h.data_ptr() for h in hidden])
                    _lib.check(self._lib.iaf_step_bwd_saved(plan, _ptr(z), _ptr(z_out), _ptr(logsd), harr,
                                                            arr([l[0] for l in layers]), arr([l[1] for l in layers]),
                                                            _ptr(g_zout), _ptr(g_logsd), _ptr(g_logdet), _ptr(g_z),
                                                            _ptr(g_ctx), pa(gw), pa(gs), pa(gb), B, _stream(dev)))
                    return g_z, g_ctx, gw, gs, gb
                _lib.check(self._lib.iaf_step_bwd(plan, _ptr(z), _ptr(context), arr([l[0] for l in layers]),
                                                  arr([l[1] for l in layers]), _ptr(g_zout), _ptr(g_logsd), _ptr(g_logdet),
                                                  _ptr(g_z), _ptr(g_ctx), pa(gw), pa(gs), pa(gb), B, _stream(dev)))
            else:
                g_outs = [torch.zeros((B, h, H, W), device=dev) if g is None else _check_input(g, "grad")
                          for g, h in zip(grads_out, self.heads)]
                go = (C.c_void_p * len(g_outs))(*[g.data_ptr() for g in g_outs])
                if saved is not None:
                    hidden = saved[2]
                    harr = (C.c_void_p * max(1, len(hidden)))(*[h.data_ptr() for h in hidden])
                    _lib.check(self._lib.iaf_multiconv_bwd_saved(plan, _ptr(z), harr, arr([l[0] for l in layers]),
                                                                 arr([l[1] for l in layers]), go, _ptr(g_z), _ptr(g_ctx),
                                                                 pa(gw), pa(gs), pa(gb), B, _stream(dev)))
                    return g_z, g_ctx, gw, gs, gb
                _lib.check(self._lib.iaf_multiconv_bwd(plan, _ptr(z), _ptr(context), arr([l[0] for l in layers]),
                                                       arr([l[1] for l in layers]), go, _ptr(g_z), _ptr(g_ctx), pa(gw),
                                                       pa(gs), pa(gb), B, _stream(dev)))
        return g_z, g_ctx, gw, gs, gb

    def step_backward(self, z, context, g_z_out, g_logsd=None, g_logdet=None, need_params=True):
        """Explicit (non-autograd) entry to iaf_step_bwd with the current weights."""
        return self._backward("step", z, context, self._layers, (g_z_out, g_logsd, g_logdet), need_params)


def _regroup(flat):
    return [tuple(flat[i:i + 3]) for i in range(0, len(flat), 3)]


def _flat_param_grads(gw, gs, gb, n_layers):
    if gw is None:
        return [None] * (3 * n_layers)
    return [t for i in range(n_layers) for t in (gw[i], gs[i], gb[i])]


class _StepFn(torch.autograd.Function):
    """autograd node of the fused step: forward = iaf_step_fwd_train (the step's own kernels also keep the hidden
    activations), backward = iaf_step_bwd_saved (no recompute)."""

    @staticmethod
    def forward(ctx, op, z, context, *flat):
        with torch.no_grad():
            z_out, logsd, logdet, hidden = op._step_train_raw(z, context)
        ctx.op = op
        ctx.has_ctx = context is not None
        ctx.n_hidden = len(hidden)
        ctx.set_materialize_grads(False)  # unused outputs arrive as None, not as zero tensors
        # the context itself is not needed by the backward (it only enters the forward); keep it as the shape template
        ctx.save_for_backward(z, *([context] if context is not None else []), z_out, logsd, *hidden, *flat)
        return z_out, logsd, logdet

    @staticmethod
    def backward(ctx, g_zout, g_logsd, g_logdet):
        saved = ctx.saved_tensors
        z = saved[0]
        context = saved[1] if ctx.has_ctx else None
        i = 2 if ctx.has_ctx else 1
        z_out, logsd = saved[i], saved[i + 1]
        hidden = list(saved[i + 2:i + 2 + ctx.n_hidden])
        flat = saved[i + 2 + ctx.n_hidden:]
        need_params = any(ctx.needs_input_grad[3:])
        g_z, g_ctx, gw, gs, gb = ctx.op._backward("step", z, context, _regroup(flat), (g_zout, g_logsd, g_logdet), need_params,
                                                   saved=(z_out, logsd, hidden))
        return (None, g_z, g_ctx) + tuple(_flat_param_grads(gw, gs, gb, len(flat) // 3))


class _LayerFn(torch.autograd.Function):
    """autograd node of the fused stochastic-layer block: forward = iaf_layer_fwd, backward = iaf_layer_bwd."""

    @staticmethod
    def forward(ctx, op, eps, post_mean, post_logsd, prior_mean, prior_logsd, context, *flat):
        with torch.no_grad():
            out = op._layer_raw(eps, post_mean, post_logsd, prior_mean, prior_logsd, context, True)
        ctx.op = op
        ctx.has_ctx = context is not None
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(eps, post_mean, post_logsd, prior_mean, prior_logsd, *([context] if context is not None else []),
                              *flat)
        return out

    @staticmethod
    def backward(ctx, g_z, g_kl, g_kl_bc, g_kl_cost):
        saved = ctx.saved_tensors
        eps, pm, pls, prm, prl = saved[:5]
        context = saved[5] if ctx.has_ctx else None
        flat = saved[6 if ctx.has_ctx else 5:]
        op = ctx.op
        layers = _regroup(flat)
        need_params = any(ctx.needs_input_grad[7:])
        eps_c, context_c, B, H, W = op._shapes(eps, context)
        dev = eps_c.device
        plan = op._plan(H, W, dev, layers)
        n = len(layers)
        arr = lambda ts: (C.c_void_p * n)(*[t.data_ptr() for t in ts])
        ts = [_check_input(t, "layer input", eps_c.shape) for t in (pm, pls, prm, prl)]
        gs_in = [None if g is None else _check_input(g, "grad") for g in (g_z, g_kl, g_kl_bc, g_kl_cost)]
        outs = [torch.empty_like(eps_c) for _ in range(5)]  # post_mean, post_logsd, prior_mean, prior_logsd, eps
        g_ctx = torch.empty_like(context_c) if context_c is not None else None
        gw = gs = gb = None
        if need_params:
            gw, gs, gb = ([torch.empty_like(l[j]) for l in layers] for j in range(3))
        pa = lambda x: arr(x) if x is not None else None
        with torch.cuda.device(dev):
            _lib.check(op._lib.iaf_layer_bwd(plan, _ptr(eps_c), _ptr(ts[0]), _ptr(ts[1]), _ptr(ts[2]), _ptr(ts[3]),
                                             _ptr(context_c), arr([l[0] for l in layers]), arr([l[1] for l in layers]),
                                             _ptr(gs_in[0]), _ptr(gs_in[1]), _ptr(gs_in[2]), _ptr(gs_in[3]),
                                             _ptr(outs[0]), _ptr(outs[1]), _ptr(outs[2]), _ptr(outs[3]), _ptr(outs[4]),
                                             _ptr(g_ctx), pa(gw), pa(gs), pa(gb), B, _stream(dev)))
        return (None, outs[4], outs[0], outs[1], outs[2], outs[3], g_ctx) + tuple(_flat_param_grads(gw, gs, gb, n))


class _MulticonvFn(torch.autograd.Function):
    """autograd node of the un-fused operator: forward = iaf_multiconv_fwd, backward = iaf_multiconv_bwd."""

    # The forward keeps the hidden activations (iaf_multiconv_fwd_train) and the backward skips the recompute
    # (iaf_multiconv_bwd_saved), as the fused step's node does (confirmed on a B200 in round 2).
    # IAF_MULTICONV_SAVED=0 falls back to recomputing them in the backward.
    @staticmethod
    def forward(ctx, op, z, context, *flat):
        ctx.keep = os.environ.get("IAF_MULTICONV_SAVED", "1") != "0"
        with torch.no_grad():
            if ctx.keep:
                outs, hidden = op._multiconv_train_raw(z, context)
            else:
                outs, hidden = op._multiconv_raw(z, context), []
        ctx.op = op
        ctx.has_ctx = context is not None
        ctx.n_hidden = len(hidden)
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(z, *([context] if context is not None else []), *hidden, *flat)
        return tuple(outs)

    @staticmethod
    def backward(ctx, *g_outs):
        saved = ctx.saved_tensors
        z = saved[0]
        context = saved[1] if ctx.has_ctx else None
        i = 2 if ctx.has_ctx else 1
        hidden = list(saved[i:i + ctx.n_hidden])
        flat = saved[i + ctx.n_hidden:]
        need_params = any(ctx.needs_input_grad[3:])
        g_z, g_ctx, gw, gs, gb = ctx.op._backward("multiconv", z, context, _regroup(flat), g_outs, need_params,
                                                   saved=(None, None, hidden) if ctx.keep else None)
        return (None, g_z, g_ctx) + tuple(_flat_param_grads(gw, gs, gb, len(flat) // 3))


# ------------------------------------------------------------------------------------
# TF-style entry: tf_utils/layers.py:158-166
# ------------------------------------------------------------------------------------
_TF_OPS = {}       # call-site key -> IAFOperator, in least-recently-used order
_TF_OPS_MAX = 256


def _tf_layers(name, params, n_h, n_out):
    """Collect V/g/b under the TF variable names ``{name}/layer_{i}/{V,g,b}`` and
    ``{name}/layer_out_{k}/...`` (layers.py:160-166, 53-55); the ``{name}/`` prefix is optional."""
    def get(scope, k):
        for key in ("%s/%s/%s" % (name, scope, k), "%s/%s" % (scope, k)):
            if key in params:
                return params[key]
        raise KeyError("parameter %s/%s/%s not found" % (name, scope, k))
    layers = [tuple(get("layer_%d" % i, k) for k in "Vgb") for i in range(len(n_h))]
    layers += [tuple(get("layer_out_%d" % i, k) for k in "Vgb") for i in range(len(n_out))]
    return layers


def _nl_name(nl):
    if callable(nl):
        nl = getattr(nl, "__name__", str(nl))
    return nl


def ar_multiconv2d(name, x, context, n_h, n_out, nl="elu", params=None, path="auto", init=False, **_):
    """Drop-in for tf_utils/layers.py:ar_multiconv2d -> list of tensors (one per n_out entry).
    ``params`` stands in for the TF variable scope: a dict holding V/g/b under the TF names.
    ``init=True`` is the data-dependent initialisation the reference runs once under ``arg_scope(..., init=True)``
    (layers.py:38-51): g and b are created in ``params`` where absent, set from this batch's statistics, and the
    init pass's outputs are returned."""
    if params is None:
        raise ValueError("params (the variable store) is required in eager mode")
    if init:
        scopes = [("layer_%d" % i, s) for i, s in enumerate(n_h)] + [("layer_out_%d" % i, s) for i, s in enumerate(n_out)]
        for scope, size in scopes:
            for k in "gb":
                if "%s/%s/%s" % (name, scope, k) not in params and "%s/%s" % (scope, k) not in params:
                    params["%s/%s/%s" % (name, scope, k)] = torch.zeros(int(size), device=x.device)
    nl = _nl_name(nl)
    # one operator (plans + packed weights) per distinct call site; the parameters are re-bound on every call, so two
    # variable stores sharing a scope name stay correct (they re-pack when they alternate) and nothing is keyed on
    # id(params), which python recycles
    key = (name, int(x.shape[1]), tuple(n_h), tuple(n_out), nl, path)
    op = _TF_OPS.pop(key, None)
    if op is None:
        op = IAFOperator("tf", x.shape[1], n_h, n_out, nl=nl, path=path)
        while len(_TF_OPS) >= _TF_OPS_MAX:
            _TF_OPS.pop(next(iter(_TF_OPS)))  # least recently used
    _TF_OPS[key] = op  # (re-)insert as most recently used
    op.set_weights(_tf_layers(name, params, n_h, n_out))
    if init:
        return op.data_init(x, context, names=["%s/layer_%d" % (name, i) for i in range(len(n_h))] +
                            ["%s/layer_out_%d" % (name, i) for i in range(len(n_out))])
    return op.multiconv(x, context)


# ------------------------------------------------------------------------------------
# Theano-style factory: graphy/nodes/ar.py:378-423
# ------------------------------------------------------------------------------------
class _Struct(object):  # graphy/__init__.py:35-39
    def __init__(self, **entries):
        self.__dict__.update(entries)

    def __call__(self, *a, **k):
        return self.__dict__["__call__"](*a, **k)


def multiconv2d(name, n_in, n_h, n_out, size_kernel=(3, 3), flipmask=False, nl="relu", w=None, device="cuda",
                path="auto"):
    """Drop-in for graphy/nodes/ar.py:multiconv2d.  Creates the parameters the reference creates
    (``{name}_{i}_w/_b/_s`` and ``{name}_out_{k}_w/_b/_s``, ar.py:288-296) in ``w`` if absent and
    returns an object with ``__call__(h, context, w, return_hiddens=False)``, ``w`` and ``postup``."""
    if w is None:
        w = {}
    if not isinstance(n_out, list) and isinstance(n_out, int):
        n_out = [n_out]
    if tuple(size_kernel) != (3, 3):
        raise NotImplementedError("only the 3x3 kernel the reference uses (train.py:63) is implemented")
    if flipmask:
        raise NotImplementedError("flipmask=True is never used on the down_iaf2_nl / up_iaf2_nl path (models.py:92)")
    sizes = [n_in] + list(n_h)
    names, masks = [], []
    specs = [(name + "_" + str(i), sizes[i], sizes[i + 1], False) for i in range(len(n_h))]
    specs += [(name + "_out_" + str(i), sizes[-1], n_out[i], True) for i in range(len(n_out))]
    for lname, cin, cout, zd in specs:
        assert cin % cout == 0 or cout % cin == 0  # ar.py:250,257
        mask = theano_conv_ar_mask(cin, cout, (3, 3), zd)
        if lname + "_w" not in w:  # ar.py:288, 293-296
            w[lname + "_w"] = torch.from_numpy(mask * 0.05 * np.random.randn(cout, cin + 1, 3, 3)).float().to(device)
            w[lname + "_b"] = torch.zeros(cout, device=device)
            w[lname + "_s"] = torch.zeros(cout, device=device)
        names.append(lname)
        masks.append(mask)
    op = IAFOperator("theano", n_in, n_h, n_out, nl=nl, path=path)

    def f(h, context, w, return_hiddens=False):
        if return_hiddens:
            raise NotImplementedError("return_hiddens=True: hidden activations never leave the SM in the fused kernel")
        op.set_weights([(w[n + "_w"], w[n + "_s"], w[n + "_b"]) for n in names])
        if "__init" in w:  # ar.py:331-353: data-dependent init, w[..._s] / w[..._b] updated in place (set_value)
            out = op.data_init(h, context, names=names)
        else:
            out = op.multiconv(h, context)
        if len(n_out) == 1:
            out = out[0]  # ar.py:411
        return out

    def postup(updates, w):
        """ar.py:369-373: re-apply the mask to an updated weight.  ``updates`` maps parameter
        name -> new value (Theano keys by shared variable; names are the eager equivalent)."""
        for n, m in zip(names, masks):
            if n + "_w" in updates:
                u = updates[n + "_w"]
                updates[n + "_w"] = u * torch.from_numpy(m).to(u.device, u.dtype)
        return updates

    return _Struct(__call__=f, w=w, postup=postup, op=op, names=names)


# ------------------------------------------------------------------------------------
# fused entry
# ------------------------------------------------------------------------------------
def iaf_step(z, context, op):
    """(z', arw_logsd_elem, logdet_per_sample) for an IAFOperator with weights set."""
    return op.step(z, context)
