"""Data-dependent initialisation of the masked-AR stack (iaf_multiconv_init / IAFOperator.data_init).

CPU: the fp64 oracle (oracle/init_oracle.py) and the C ABI under host emulation (tests/emu) against the fixture produced
by executing the reference's own init branches (tests/golden/make_golden_init.py), determinism, argument checks, the
python front-ends over the emulated library, and the init kernels under ThreadSanitizer / AddressSanitizer+UBSan.
GPU: the same fixture cases and seeded shapes on the device, every path, and what a forward does with the new
parameters.  Metric: ||delta||_inf / max(||ref||_inf, 1) <= 1e-4 for the outputs and for every new parameter.
"""
import contextlib
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

from iaf_b200 import _lib as L
from oracle import iaf_oracle as O
from oracle import init_oracle as IO
from tests.golden.make_golden_init import INIT_CASES

HERE = os.path.dirname(os.path.abspath(__file__))
TOL = 1e-4
CASE_IDS = [c[0] for c in INIT_CASES]


def rel(a, ref):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    ref = np.asarray(ref, dtype=np.float64)
    assert np.isfinite(a).all()
    return float(np.abs(a.astype(np.float64) - ref).max() / max(np.abs(ref).max(), 1.0))


def keys(variant):
    return ("V", "g", "b") if variant == "tf" else ("w", "s", "b")


def fixture(name):
    g = np.load(os.path.join(HERE, "golden", "data_init.npz"))
    case = INIT_CASES[CASE_IDS.index(name)]
    variant, hidden = case[1], case[4]
    n = len(hidden) + 2
    layers = [{k: g["%s/in/%d/%s" % (name, i, k)] for k in keys(variant)} for i in range(n)]
    ref = dict(outs=[g["%s/out/%d" % (name, k)] for k in range(2)],
               scale=[g["%s/scale/%d" % (name, i)] for i in range(n)], bias=[g["%s/bias/%d" % (name, i)] for i in range(n)])
    return case, layers, g[name + "/z"], g[name + "/ctx"], ref


def oracle(variant, z, ctx, layers, n_hidden, nl):
    f64 = [{k: v.astype(np.float64) for k, v in l.items()} for l in layers]
    return IO.data_init(variant, z.astype(np.float64), ctx.astype(np.float64), f64[:n_hidden], f64[n_hidden:], nl)


# ---------------------------------------------------------------------------------------
# the oracle against the reference's own init branches
# ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", CASE_IDS)
def test_oracle_matches_reference_fixture(name):
    (_, variant, _, _, hidden, _, _, nl), layers, z, ctx, ref = fixture(name)
    outs, params, zeros = oracle(variant, z, ctx, layers, len(hidden), nl)
    for o, r in zip(outs, ref["outs"]):
        assert rel(o, r) < 1e-10
    for (s, b), rs, rb in zip(params, ref["scale"], ref["bias"]):
        assert rel(s, rs) < 1e-10 and rel(b, rb) < 1e-10
    assert (sum(zeros) > 0) == (name == "th_skip")


def test_fixture_covers_the_quirks():
    """The cases exercise what the issue pins: the 1e5 scale of a zero TF column, the skipped Theano layer, and the TF
    parameters for which a forward does NOT reproduce the init output (exp(g) vs exp(3g))."""
    (_, _, _, _, hidden, _, _, _), layers, z, ctx, ref = fixture("tf_zero_col")
    assert abs(ref["scale"][0][3] - np.log(1e5) / 3.0) < 1e-9 and ref["bias"][0][3] == 0.0
    (_, _, _, _, hidden, _, _, _), layers, z, ctx, ref = fixture("th_skip")
    assert np.array_equal(ref["scale"][-1], layers[-1]["s"]) and np.array_equal(ref["bias"][-1], layers[-1]["b"])
    assert not np.array_equal(ref["scale"][-2], layers[-2]["s"])
    (_, variant, _, _, hidden, _, _, nl), layers, z, ctx, ref = fixture("tf_8_8")
    new = [dict(V=l["V"].astype(np.float64), g=s, b=b) for l, s, b in zip(layers, ref["scale"], ref["bias"])]
    fwd = O.multiconv("tf", z.astype(np.float64), ctx.astype(np.float64), new[:2], new[2:], nl)
    assert rel(fwd[0], ref["outs"][0]) > 1e-2


# ---------------------------------------------------------------------------------------
# the C ABI under host emulation
# ---------------------------------------------------------------------------------------
def _emu_plan(variant, n_z, hidden, H, W, nl):
    from tests.emu.harness import emu
    lib = emu()
    d = L.IafDesc()
    d.variant, d.n_z, d.n_hidden, d.n_heads = L.VARIANTS[variant], n_z, len(hidden), 2
    for i, h in enumerate(hidden):
        d.hidden[i] = h
    d.head[0] = d.head[1] = n_z
    d.H, d.W, d.nl, d.path = H, W, L.NLS[nl], L.PATHS["simt"]
    plan = C.c_void_p()
    assert lib.iaf_plan_create(C.byref(plan), C.byref(d)) == 0
    return lib, plan


def _arr(arrays):
    return (C.c_void_p * len(arrays))(*[a.ctypes.data for a in arrays]) if arrays is not None else None


def _p(a):
    return C.c_void_p(a.ctypes.data) if a is not None else C.c_void_p(0)


def emu_init(lib, plan, variant, layers, z, ctx, n_z, pass_current=True):
    """iaf_multiconv_init on numpy buffers -> (status, outs, scales, biases, skipped)."""
    B, _, H, W = z.shape
    f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)
    ws = [f32(l[keys(variant)[0]]) for l in layers]
    ss = [f32(l[keys(variant)[1]]) for l in layers]
    bs = [f32(l[keys(variant)[2]]) for l in layers]
    so = [np.full_like(s, np.nan) for s in ss]
    bo = [np.full_like(b, np.nan) for b in bs]
    outs = [np.full((B, n_z, H, W), np.nan, np.float32) for _ in range(2)]
    skipped = np.full(len(layers), -1, np.int32)
    cur = pass_current or variant == "theano"
    z, ctx = f32(z), (f32(ctx) if ctx is not None else None)
    st = lib.iaf_multiconv_init(plan, _p(z), _p(ctx), _arr(ws), _arr(ss) if cur else None,
                                _arr(bs) if cur else None, _arr(so), _arr(bo), _arr(outs), _p(skipped), B, None)
    return st, outs, so, bo, skipped


@pytest.mark.parametrize("name", CASE_IDS)
def test_emulated_abi_matches_fixture_and_oracle(name):
    (_, variant, B, n_z, hidden, H, W, nl), layers, z, ctx, ref = fixture(name)
    lib, plan = _emu_plan(variant, n_z, hidden, H, W, nl)
    try:
        st, outs, so, bo, skipped = emu_init(lib, plan, variant, layers, z, ctx if hidden else None, n_z,
                                             pass_current=(variant == "theano"))
        assert st == 0
        o_outs, o_params, o_zeros = oracle(variant, z, ctx, layers, len(hidden), nl)
        for o, r, orc in zip(outs, ref["outs"], o_outs):
            assert rel(o, r) <= TOL and rel(o, orc) <= TOL
        for i in range(len(layers)):
            for got, r, orc in ((so[i], ref["scale"][i], o_params[i][0]), (bo[i], ref["bias"][i], o_params[i][1])):
                assert rel(got, r) <= TOL and rel(got, orc) <= TOL, (name, i)
        assert skipped.tolist() == o_zeros
        # reruns are bit-identical; and after the pass the plan is not packed
        st2, outs2, so2, bo2, sk2 = emu_init(lib, plan, variant, layers, z, ctx if hidden else None, n_z)
        assert st2 == 0 and np.array_equal(sk2, skipped)
        for a, b in zip(outs + so + bo, outs2 + so2 + bo2):
            assert np.array_equal(a, b)
        res = [np.empty((B, n_z, H, W), np.float32) for _ in range(2)]
        assert lib.iaf_multiconv_fwd(plan, _p(z), _p(ctx), _arr(res), B, None) == L.ERR_NOT_PACKED
    finally:
        lib.iaf_plan_destroy(plan)


def test_emulated_theano_forward_with_new_parameters_reproduces_init():
    """Theano starting from the zeros multiconv2d creates: s, b are overwritten, so the forward with the new parameters
    equals the init outputs, and every head channel has mean 0 and std 1."""
    from tests.emu.harness import EmuOperator
    n_z, hidden, H, W, B = 4, [8], 5, 6, 3
    hid, heads = O.make_params("theano", n_z, hidden, [n_z, n_z], seed=5)
    for l in hid + heads:
        l["s"][:] = 0.0
        l["b"][:] = 0.0
    z, ctx = O.make_inputs(B, n_z, hidden[0], H, W, seed=6)
    lib, plan = _emu_plan("theano", n_z, hidden, H, W, "elu")
    try:
        st, outs, so, bo, skipped = emu_init(lib, plan, "theano", hid + heads, z, ctx, n_z)
        assert st == 0 and not skipped.any()
    finally:
        lib.iaf_plan_destroy(plan)
    new = [(l["w"], s, b) for l, s, b in zip(hid + heads, so, bo)]
    fwd = EmuOperator("theano", n_z, hidden, [n_z, n_z], H, W).set_weights(new).multiconv(z, ctx)
    for f, o in zip(fwd, outs):
        assert rel(f, o) <= TOL
        assert np.abs(o.mean(axis=(0, 2, 3))).max() < 1e-5 and np.abs(o.std(axis=(0, 2, 3)) - 1).max() < 1e-4


def test_emulated_abi_argument_checks():
    (_, variant, B, n_z, hidden, H, W, nl), layers, z, ctx, ref = fixture("th_8")
    lib, plan = _emu_plan(variant, n_z, hidden, H, W, nl)
    try:
        f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)
        ws, ss, bs = ([f32(l[k]) for l in layers] for k in keys(variant))
        so, bo = [np.zeros_like(s) for s in ss], [np.zeros_like(b) for b in bs]
        good = dict(plan=plan, z=_p(z), ctx=_p(ctx), w=_arr(ws), s=_arr(ss), b=_arr(bs), so=_arr(so), bo=_arr(bo),
                    outs=None, skipped=C.c_void_p(0), B=B)

        def call(**kw):
            a = dict(good, **kw)
            return lib.iaf_multiconv_init(a["plan"], a["z"], a["ctx"], a["w"], a["s"], a["b"], a["so"], a["bo"],
                                          a["outs"], a["skipped"], a["B"], None)
        assert call() == 0                                             # outs and skipped are optional
        assert call(plan=None) == L.ERR_BAD_ARG
        assert call(z=C.c_void_p(0)) == L.ERR_BAD_ARG
        assert call(ctx=C.c_void_p(0)) == L.ERR_BAD_ARG                 # a hidden layer needs the context
        assert call(w=None) == L.ERR_BAD_ARG
        assert call(s=None) == L.ERR_BAD_ARG                            # Theano reads the current s and b
        assert call(so=None) == L.ERR_BAD_ARG and call(bo=None) == L.ERR_BAD_ARG
        assert call(B=0) == L.ERR_BAD_ARG
        assert call(so=_arr(ss)) == L.ERR_BAD_ARG                       # outputs must not alias inputs
        holes = (C.c_void_p * len(ws))(*([a.ctypes.data for a in ws[:-1]] + [0]))
        assert call(w=holes) == L.ERR_BAD_ARG
        outs1 = (C.c_void_p * 2)(np.zeros((B, n_z, H, W), np.float32).ctypes.data, 0)
        assert call(outs=outs1) == L.ERR_BAD_ARG                        # both heads or none
    finally:
        lib.iaf_plan_destroy(plan)
    # TF: the current g and b are not read and may be NULL
    (_, variant, B, n_z, hidden, H, W, nl), layers, z, ctx, ref = fixture("tf_zero_col")
    lib, plan = _emu_plan(variant, n_z, hidden, H, W, nl)
    try:
        st, outs, so, bo, skipped = emu_init(lib, plan, variant, layers, z, ctx, n_z, pass_current=False)
        assert st == 0 and not skipped.any()
        assert rel(so[0], ref["scale"][0]) <= TOL
    finally:
        lib.iaf_plan_destroy(plan)


# ---------------------------------------------------------------------------------------
# python front-ends over the emulated library
# ---------------------------------------------------------------------------------------
@pytest.fixture
def emulated_ops(monkeypatch):
    """iaf_b200.ops with its ctypes binding pointed at the emulated library and CPU tensors let through (test-only: the
    product refuses CPU tensors, see tests/test_host_cpu.py)."""
    from iaf_b200 import ops
    from tests.emu.harness import emu

    def check_input(t, name, shape=None):
        assert isinstance(t, torch.Tensor) and t.dtype == torch.float32
        if shape is not None:
            assert tuple(t.shape) == tuple(shape)
        return t.contiguous()

    monkeypatch.setattr(L, "lib", emu)
    monkeypatch.setattr(ops, "_check_input", check_input)
    monkeypatch.setattr(ops, "_stream", lambda device: C.c_void_p(0))
    monkeypatch.setattr(torch.cuda, "device", lambda d: contextlib.nullcontext())
    return ops


def test_python_data_init_over_the_emulated_abi(emulated_ops):
    ops = emulated_ops
    (_, variant, B, n_z, hidden, H, W, nl), layers, z, ctx, ref = fixture("th_8")
    params = [tuple(torch.from_numpy(l[k].copy()).requires_grad_(True) for k in keys(variant)) for l in layers]
    op = ops.IAFOperator(variant, n_z, hidden, [n_z, n_z], nl=nl, path="simt").set_weights(params)
    zt, ct = torch.from_numpy(z), torch.from_numpy(ctx)
    before = op.multiconv(zt, ct)[0].detach().clone()          # packs the plan with the old parameters
    versions = [(s._version, b._version) for _, s, b in params]
    outs = op.data_init(zt, ct)
    for o, r in zip(outs, ref["outs"]):
        assert rel(o, r) <= TOL and not o.requires_grad
    for i, (_, s, b) in enumerate(params):
        assert rel(s.detach(), ref["scale"][i]) <= TOL and rel(b.detach(), ref["bias"][i]) <= TOL
        assert s._version > versions[i][0] and b._version > versions[i][1]  # updated in place
    # the next call re-packs from the new parameters
    after = op.multiconv(zt, ct)[0].detach()
    new = [dict(w=l["w"].astype(np.float64), s=s.astype(np.float64), b=b.astype(np.float64))
           for l, s, b in zip(layers, ref["scale"], ref["bias"])]
    expect = O.multiconv("theano", z.astype(np.float64), ctx.astype(np.float64), new[:1], new[1:], nl)[0]
    assert rel(after, expect) <= TOL and rel(before, expect) > 1e-2


def test_python_theano_factory_init_and_skip_warning(emulated_ops):
    ops = emulated_ops
    (_, variant, B, n_z, hidden, H, W, nl), layers, z, ctx, ref = fixture("th_skip")
    w = {}
    mc = ops.multiconv2d("q", n_z, hidden, [n_z, n_z], nl=nl, w=w, device="cpu")
    for nm, l in zip(mc.names, layers):
        for k in "wsb":
            w[nm + "_" + k] = torch.from_numpy(l[k].copy())
    held = {k: v for k, v in w.items()}
    mc(torch.from_numpy(z), torch.from_numpy(ctx), w)  # packs the plan with the old parameters
    w["__init"] = True
    with pytest.warns(RuntimeWarning, match=r"Stdev=0 for 1 features in q_out_1\. Skipping data-dependent init\."):
        out = mc(torch.from_numpy(z), torch.from_numpy(ctx), w)
    for o, r in zip(out, ref["outs"]):
        assert rel(o, r) <= TOL
    for i, nm in enumerate(mc.names):
        assert w[nm + "_s"] is held[nm + "_s"] and w[nm + "_b"] is held[nm + "_b"]  # set_value: the same tensors
        assert rel(w[nm + "_s"], ref["scale"][i]) <= TOL and rel(w[nm + "_b"], ref["bias"][i]) <= TOL
    # without '__init' the factory is the plain forward again, re-packed with the new parameters
    del w["__init"]
    again = mc(torch.from_numpy(z), torch.from_numpy(ctx), w)
    new = [dict(w=l["w"].astype(np.float64), s=s, b=b) for l, s, b in zip(layers, ref["scale"], ref["bias"])]
    expect = O.multiconv("theano", z.astype(np.float64), ctx.astype(np.float64), new[:1], new[1:], nl)
    assert rel(again[0], expect[0]) <= TOL and rel(again[1], expect[1]) <= TOL


def test_python_tf_init_creates_g_b(emulated_ops):
    ops = emulated_ops
    (_, variant, B, n_z, hidden, H, W, nl), layers, z, ctx, ref = fixture("tf_8_8")
    params = {"amc/layer_%d/V" % i: torch.from_numpy(l["V"].copy()) for i, l in enumerate(layers[:2])}
    params.update({"amc/layer_out_%d/V" % k: torch.from_numpy(l["V"].copy()) for k, l in enumerate(layers[2:])})
    outs = ops.ar_multiconv2d("amc", torch.from_numpy(z), torch.from_numpy(ctx), hidden, [n_z, n_z], nl="elu",
                              params=params, path="simt", init=True)
    for o, r in zip(outs, ref["outs"]):
        assert rel(o, r) <= TOL
    scopes = ["layer_0", "layer_1", "layer_out_0", "layer_out_1"]
    for i, s in enumerate(scopes):
        assert rel(params["amc/%s/g" % s], ref["scale"][i]) <= TOL and rel(params["amc/%s/b" % s], ref["bias"][i]) <= TOL
        assert params["amc/%s/g" % s].device == torch.device("cpu")
    # existing g, b are updated in place, not replaced; init=False is the plain forward with them
    g0 = params["amc/layer_0/g"]
    ops.ar_multiconv2d("amc", torch.from_numpy(z), torch.from_numpy(ctx), hidden, [n_z, n_z], params=params, path="simt",
                       init=True)
    assert params["amc/layer_0/g"] is g0
    fwd = ops.ar_multiconv2d("amc", torch.from_numpy(z), torch.from_numpy(ctx), hidden, [n_z, n_z], params=params,
                             path="simt")
    new = [dict(V=l["V"].astype(np.float64), g=s, b=b) for l, s, b in zip(layers, ref["scale"], ref["bias"])]
    assert rel(fwd[0], O.multiconv("tf", z.astype(np.float64), ctx.astype(np.float64), new[:2], new[2:])[0]) <= TOL


# ---------------------------------------------------------------------------------------
# sanitizers over the init kernels
# ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("san", ["thread", "address,undefined"])
def test_init_kernels_under_sanitizers(tmp_path, san):
    """tests/emu/init_check.cc: iaf_multiconv_init (pack, layer conv, statistics, finalize, apply) on a Theano stack with
    a skipped head, a TF stack and a no-hidden-layer stack, with ThreadSanitizer (one std::thread per CUDA thread, a
    std::barrier per __syncthreads: a missing barrier is a reported race) and with AddressSanitizer + UBSan."""
    csrc = os.path.join(os.path.dirname(HERE), "iaf_b200", "csrc")
    emu_dir = os.path.join(HERE, "emu")
    exe = str(tmp_path / "init_check")
    cmd = ["g++", "-std=c++20", "-O1", "-g", "-fsanitize=" + san, "-fno-sanitize-recover=undefined", "-pthread", "-DIAF_EMU",
           "-w", "-I", emu_dir, "-I", csrc]
    for f in ("iaf_capi.cu", "iaf_pack.cu", "iaf_simt.cu", "iaf_bwd.cu"):
        cmd += ["-x", "c++", os.path.join(csrc, f)]
    cmd += ["-x", "c++", os.path.join(emu_dir, "tc_stub.cc"), "-x", "c++", os.path.join(emu_dir, "init_check.cc"), "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0 and ("san" in (r.stderr + r.stdout).lower() and "cannot find" in (r.stderr + r.stdout).lower()):
        pytest.skip("sanitizer runtime not available: " + r.stderr[-200:])
    assert r.returncode == 0, r.stderr[-2000:]
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, TSAN_OPTIONS="halt_on_error=0 exitcode=66", ASAN_OPTIONS="detect_leaks=0"))
    assert "Sanitizer" not in r.stderr and "runtime error" not in r.stderr, r.stderr[:3000]
    assert r.returncode == 0 and "init_check ok" in r.stdout, (r.returncode, r.stdout[-500:], r.stderr[-500:])


# ---------------------------------------------------------------------------------------
# on the B200
# ---------------------------------------------------------------------------------------
def gpu_op(variant, n_z, hidden, layers, nl="elu", path="auto"):
    from iaf_b200 import IAFOperator
    ts = [tuple(torch.from_numpy(np.ascontiguousarray(l[k], dtype=np.float32)).cuda() for k in keys(variant)) for l in layers]
    return IAFOperator(variant, n_z, hidden, [n_z, n_z], nl=nl, path=path).set_weights(ts), ts


def gpu_paths(variant, n_z, hidden, H, W):
    """auto and simt always; tc where a plan accepts the shape."""
    from iaf_b200 import IAFOperator
    paths = ["auto", "simt"]
    hid, heads = O.make_params(variant, n_z, hidden, [n_z, n_z], seed=0)
    try:
        gpu_op(variant, n_z, hidden, hid + heads, path="tc")[0].path_used(H, W, "cuda:0")
        paths.append("tc")
    except NotImplementedError:
        pass
    return paths


def gpu_init(variant, n_z, hidden, layers, z, ctx, nl="elu", path="auto"):
    op, ts = gpu_op(variant, n_z, hidden, layers, nl, path)
    outs = op.data_init(torch.from_numpy(z).cuda(), torch.from_numpy(ctx).cuda() if hidden else None)
    torch.cuda.synchronize()
    return op, ts, outs


def check_against(outs, ts, ref_outs, ref_params, tag):
    for o, r in zip(outs, ref_outs):
        assert rel(o, r) <= TOL, tag
    for i, (t, (s, b)) in enumerate(zip(ts, ref_params)):
        assert rel(t[1], s) <= TOL and rel(t[2], b) <= TOL, (tag, i)


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASE_IDS)
def test_gpu_fixture_cases_on_every_path(name):
    (_, variant, B, n_z, hidden, H, W, nl), layers, z, ctx, ref = fixture(name)
    results = {}
    for path in gpu_paths(variant, n_z, hidden, H, W):
        if name == "th_skip":
            with pytest.warns(RuntimeWarning, match="Stdev=0 for 1 features in layer_out_1"):
                op, ts, outs = gpu_init(variant, n_z, hidden, layers, z, ctx, nl, path)
        else:
            op, ts, outs = gpu_init(variant, n_z, hidden, layers, z, ctx, nl, path)
        check_against(outs, ts, ref["outs"], list(zip(ref["scale"], ref["bias"])), (name, path))
        results[path] = [t.cpu() for t in outs] + [t.cpu() for l in ts for t in l[1:]]
    for path, r in results.items():  # the same exact-fp32 kernels on every plan: bit-identical
        assert all(torch.equal(a, b) for a, b in zip(r, results["simt"])), path


SEEDED = [
    # tag, variant, B, n_z, hidden, H, W, nl
    ("C1_16", "theano", 16, 32, [64], 16, 16, "elu"),
    ("C1_8", "theano", 16, 32, [64], 8, 8, "elu"),
    ("C1_4", "theano", 16, 32, [64], 4, 4, "elu"),
    ("C2a_B16", "tf", 16, 32, [64], 16, 16, "elu"),
    ("C2a_B256", "tf", 256, 32, [64], 16, 16, "elu"),
    ("C2b_B32", "tf", 32, 32, [160, 160], 16, 16, "elu"),
    ("C4_8", "theano", 8, 32, [160, 160], 8, 8, "softplus"),
    ("depth0", "theano", 8, 32, [], 16, 16, "elu"),
    ("simt_only", "tf", 4, 6, [12], 7, 5, "elu"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("tag,variant,B,n_z,hidden,H,W,nl", SEEDED, ids=[c[0] for c in SEEDED])
def test_gpu_seeded_shapes_against_oracle(tag, variant, B, n_z, hidden, H, W, nl):
    hid, heads = O.make_params(variant, n_z, hidden, [n_z, n_z], seed=3)
    z, ctx = O.make_inputs(B, n_z, hidden[0] if hidden else n_z, H, W, seed=4)
    op, ts, outs = gpu_init(variant, n_z, hidden, hid + heads, z, ctx, nl)
    ref_outs, ref_params, zeros = oracle(variant, z, ctx, hid + heads, len(hidden), nl)
    assert not any(zeros)
    check_against(outs, ts, ref_outs, ref_params, tag)


@pytest.mark.gpu
def test_gpu_paths_give_bit_identical_results():
    variant, B, n_z, hidden, H, W = "tf", 16, 32, [64], 16, 16
    hid, heads = O.make_params(variant, n_z, hidden, [n_z, n_z], seed=8)
    z, ctx = O.make_inputs(B, n_z, hidden[0], H, W, seed=9)
    paths = gpu_paths(variant, n_z, hidden, H, W)
    assert "tc" in paths
    res = {}
    for path in paths:
        op, ts, outs = gpu_init(variant, n_z, hidden, hid + heads, z, ctx, path=path)
        res[path] = [o.cpu() for o in outs] + [t.cpu() for l in ts for t in l[1:]]
        again = op.data_init(torch.from_numpy(z).cuda(), torch.from_numpy(ctx).cuda())  # g, b are not read: same result
        assert all(torch.equal(a.cpu(), b) for a, b in zip(again, res[path][:2]))
    for path in paths:
        assert all(torch.equal(a, b) for a, b in zip(res[path], res["simt"])), path


@pytest.mark.gpu
@pytest.mark.parametrize("H", [16, 8])
def test_gpu_theano_from_factory_zeros_forward_reproduces_init(H):
    """multiconv2d creates s = b = 0; the init pass overwrites them, so the forward with the new parameters on the same
    batch reproduces the init outputs on whichever path the plan uses, and each head channel has mean 0, std 1."""
    from iaf_b200 import multiconv2d
    np.random.seed(12)
    B, n_z, hidden = 16, 32, [64]
    w = {}
    mc = multiconv2d("q", n_z, hidden, [n_z, n_z], nl="elu", w=w)
    z, ctx = O.make_inputs(B, n_z, hidden[0], H, H, seed=13)
    zt, ct = torch.from_numpy(z).cuda(), torch.from_numpy(ctx).cuda()
    w["__init"] = True
    outs = mc(zt, ct, w)
    del w["__init"]
    fwd = mc(zt, ct, w)
    for o, f in zip(outs, fwd):
        assert rel(f, o.cpu().numpy().astype(np.float64)) <= TOL, mc.op.path_used(H, H, "cuda:0")
        o64 = o.double()
        assert float(o64.mean(dim=(0, 2, 3)).abs().max()) < 1e-5
        assert float((o64.std(dim=(0, 2, 3), unbiased=False) - 1).abs().max()) < 1e-4


@pytest.mark.gpu
def test_gpu_tf_forward_with_new_parameters_is_not_the_init_output():
    """TF: the forward uses exp(g) where the init pass scaled by exp(3g) (layers.py:60 vs 47): the new parameters' forward
    matches the oracle forward with those parameters, and not the init outputs."""
    variant, B, n_z, hidden, H, W = "tf", 16, 32, [64], 16, 16
    hid, heads = O.make_params(variant, n_z, hidden, [n_z, n_z], seed=14)
    z, ctx = O.make_inputs(B, n_z, hidden[0], H, W, seed=15)
    op, ts, outs = gpu_init(variant, n_z, hidden, hid + heads, z, ctx)
    fwd = op.multiconv(torch.from_numpy(z).cuda(), torch.from_numpy(ctx).cuda())
    new = [dict(V=l["V"].astype(np.float64), g=t[1].double().cpu().numpy(), b=t[2].double().cpu().numpy())
           for l, t in zip(hid + heads, ts)]
    ref = O.multiconv("tf", z.astype(np.float64), ctx.astype(np.float64), new[:1], new[1:])
    for f, r, o in zip(fwd, ref, outs):
        assert rel(f, r) <= TOL
        assert rel(f, o.cpu().numpy().astype(np.float64)) > 1e-2


@pytest.mark.gpu
def test_gpu_step_after_init_uses_new_parameters_and_plan_is_unpacked():
    variant, B, n_z, hidden, H, W = "theano", 8, 32, [64], 8, 8
    hid, heads = O.make_params(variant, n_z, hidden, [n_z, n_z], seed=16)
    z, ctx = O.make_inputs(B, n_z, hidden[0], H, W, seed=17)
    op, ts = gpu_op(variant, n_z, hidden, hid + heads)
    zt, ct = torch.from_numpy(z).cuda(), torch.from_numpy(ctx).cuda()
    old = op.step(zt, ct)[0].cpu()
    op.data_init(zt, ct)
    plan = op._plans[(H, W, 0)][0]
    outs = [torch.empty((B, n_z, H, W), device="cuda") for _ in range(2)]
    arr = (C.c_void_p * 2)(*[o.data_ptr() for o in outs])
    # at the C level the plan is not packed until iaf_pack_weights runs again
    assert op._lib.iaf_multiconv_fwd(plan, C.c_void_p(zt.data_ptr()), C.c_void_p(ct.data_ptr()), arr, B, None) == \
        L.ERR_NOT_PACKED
    z1, _, logdet = op.step(zt, ct)  # re-packs
    new = [dict(w=l["w"].astype(np.float64), s=t[1].double().cpu().numpy(), b=t[2].double().cpu().numpy())
           for l, t in zip(hid + heads, ts)]
    zr, _, ldr = O.iaf_step("theano", z.astype(np.float64), ctx.astype(np.float64), new[:1], new[1:])
    assert rel(z1, zr) <= TOL and rel(logdet, ldr) <= TOL
    assert rel(old, zr) > 1e-3
    assert op._lib.iaf_multiconv_fwd(plan, C.c_void_p(zt.data_ptr()), C.c_void_p(ct.data_ptr()), arr, B, None) == 0
