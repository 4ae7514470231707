#!/usr/bin/env python
"""bench.py -- IAF-transform throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c2a|c2b|...] [--dump-outputs DIR]

A "step" is one fused IAF step (masked-AR conv stack -> mu, s -> z' = (z - .1 mu)/exp(.1 s),
per-element arw_logsd, per-sample logdet) over one GLOBAL batch of 256 synthetic samples of
n_z=32, 16x16 (SURVEY 8d).  Metric: latent elements/s = 256*n_z*H*W / t_step, whole job.

* value      : inputs resident in HBM.  The K steps are grouped into ELBO evaluations of E steps
               (E = the number of IAF steps per ELBO of the model the workload comes from); each group
               is one CUDA-graph replay (the E step launches, then the ELBO scalar = the sum of the
               group's log-dets, captured in the same graph; at N = 1 all groups form one graph) and, at N > 1, ONE all-reduce of that scalar (tf_train.py:142), issued on a side stream so it
               overlaps the next group's kernels.  CUDA events around the whole region, max over ranks.
               The steps rotate through NSETS input/output sets whose footprint exceeds L2.
* roofline   : the step kernel(s) alone: one CUDA graph of K back-to-back launches, CUDA events;
               bound = whichever of algorithmic-bytes/HBM-peak and algorithmic-flops/bf16-peak is larger.
* e2e        : same metric through the public host-buffer entry (IAFOperator.submit_host ->
               iaf_step_submit_host): pinned host inputs H2D, step, results D2H, every step,
               pipelined over three device staging slots; timed until wait_host() returns.
* also       : the other headline shape (hidden [160,160]: c2b at N=1, the same batch sharded = c5 at N>1),
               device-timed in the same run; at N=1 also `training_pair`: forward keeping the activations
               + backward from them (all gradients) for both shapes, microseconds per call.
* cpu_baseline / --impl reference: the oracle's torch-CPU port of the reference path on this box's
               cores (the reference's Theano/TF code cannot run in this image; SURVEY F4).  ONE routine
               serves both: per thread-count candidate 3 warm-up + 5 timed calls (median), the best
               candidate then runs the timed steps; the b200 arm runs it in a fresh subprocess so that
               both arms measure under the same conditions.

N>1: launched by torchrun, one rank per GPU; the GLOBAL batch of 256 is sharded (256/N samples per rank:
strong scaling, north_star / SURVEY 8e), weights replicated, no data-path collective.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402,F401
import torch  # noqa: E402

GLOBAL_B = 256
WORKLOADS = {
    # name: (variant, n_z, hidden, H, W, global batch, IAF steps per ELBO evaluation of the model it comes from)
    "c2a": ("tf", 32, [64], 16, 16, GLOBAL_B, 6),               # hidden [64]: README cifar10 model, depths [2,2,2] -> 6 steps/ELBO
    "c2b": ("tf", 32, [160, 160], 16, 16, GLOBAL_B, 20),        # hidden [160,160]: tf_train.py, num_blocks=20 x depth=1
    # per-step shapes of the other BASELINE configs (parity-test cases; benched for the record, not the headline)
    "c1": ("theano", 32, [64], 16, 16, 16, 6),                  # README example, batch 16, level 0
    "c1_l1": ("theano", 32, [64], 8, 8, 16, 6),                 # ... level 1
    "c1_l2": ("theano", 32, [64], 4, 4, 16, 6),                 # ... level 2
    "c3": ("tf", 32, [160, 160], 16, 16, 32, 20),               # tf_train.py default per-GPU batch
    "c4_l1": ("theano", 32, [160, 160], 8, 8, 16, 20),          # Table-3 config, second level
}
METRIC = "IAF latents/sec (z',logdet) @ n_z=32,16x16,bs256"
UNIT = "latent elements/s"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), "measured (MEASURED_PEAKS.json, burst)"
    return 6650.0, 1590.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------
# host topology: physical cores, NUMA nodes, the GPU's local CPUs
# ----------------------------------------------------------------------------------------------
def _parse_cpulist(s):
    out = set()
    for part in s.strip().split(","):
        if not part:
            continue
        if "-" in part:
            a, b = part.split("-")
            out.update(range(int(a), int(b) + 1))
        else:
            out.add(int(part))
    return out


def host_topology():
    """(allowed cpus, physical cores among them, physical cores of the largest NUMA node among them)."""
    allowed = set(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else set(range(os.cpu_count() or 1))
    phys = set()
    for c in sorted(allowed):
        try:
            with open("/sys/devices/system/cpu/cpu%d/topology/thread_siblings_list" % c) as f:
                sib = _parse_cpulist(f.read())
            phys.add(min(sib & allowed) if sib & allowed else c)
        except OSError:
            phys.add(c)
    node_phys = 0
    try:
        for n in os.listdir("/sys/devices/system/node"):
            if n.startswith("node") and n[4:].isdigit():
                with open("/sys/devices/system/node/%s/cpulist" % n) as f:
                    node_phys = max(node_phys, len(_parse_cpulist(f.read()) & phys))
    except OSError:
        pass
    return allowed, len(phys), node_phys or len(phys)


def bind_to_gpu_numa(index):
    """Pin this process (and therefore the pinned host buffers it allocates afterwards) to the CPUs NVML reports as
    local to GPU ``index``.  Returns a short description for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {w * 64 + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
        allowed = set(os.sched_getaffinity(0))
        cpus &= allowed
        if cpus and cpus != allowed:
            os.sched_setaffinity(0, cpus)
            return "bound to %d CPUs local to GPU %d (NVML cpu affinity)" % (len(cpus), index)
        return "GPU %d is local to every allowed CPU (%d): no binding needed" % (index, len(allowed))
    except Exception as e:  # pragma: no cover
        return "not bound (%s)" % type(e).__name__


class ClockSampler(object):
    """Polls SM clock / throttle reasons through NVML while the timed regions run."""

    def __init__(self, index):
        self.samples = []
        self.phase = "idle"
        self.stop = False
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # pragma: no cover
            self.err = repr(e)
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self.nv
        while not self.stop:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((self.phase, mhz, reasons))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.ok:
            self.t.start()

    def finish(self):
        self.stop = True
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "NVML unavailable"}
        self.t.join(timeout=1.0)
        names = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
                 0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
                 0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}
        timed = [s for s in self.samples if s[0] == "timed"]
        window = "timed regions"
        if len(timed) < 3:
            timed = [s for s in self.samples if s[0] in ("timed", "e2e", "warmup")]
            window = "warmup+timed+e2e (timed regions shorter than 3 samples)"
        if not timed:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "no samples"}
        bits = 0
        for s in timed:
            bits |= s[2]
        reasons = [n for b, n in names.items() if bits & b and n != "gpu_idle"]
        return {"sm_mhz": statistics.median(s[1] for s in timed), "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(timed), "window": window}


def workload_string(name, world=1):
    variant, n_z, hidden, H, W, B, E = WORKLOADS[name]
    return "%s: single IAF step, n_z=%d hidden=%s %dx%d global batch %d, %s-variant numerics" % (
        name, n_z, hidden, H, W, B, variant)


def make_layers(name, seed=0):
    """Seeded synthetic (direction, gain, bias) per conv in the variant's own layout: TF V[3,3,Cin,Cout], g, b
    (layers.py:53-55); Theano w[Cout,Cin+1,3,3], s, b (ar.py:288-296; its gain is exp(3 s))."""
    variant, n_z, hidden = WORKLOADS[name][:3]
    g = torch.Generator().manual_seed(seed + 1)
    sizes = [n_z] + hidden
    layers = []
    for i in range(len(hidden) + 2):
        cin = sizes[min(i, len(hidden))]
        cout = hidden[i] if i < len(hidden) else n_z
        shape = (3, 3, cin, cout) if variant == "tf" else (cout, cin + 1, 3, 3)
        V = 0.05 * torch.randn(shape, generator=g)
        gg = torch.rand((cout,), generator=g) - 0.5
        if variant == "theano":
            gg = gg / 3.0
        b = 0.1 * torch.randn((cout,), generator=g)
        layers.append((V, gg, b))
    return layers


def make_workload(name, device, nsets, seed=0, B=None):
    from iaf_b200 import IAFOperator
    variant, n_z, hidden, H, W, Bg, E = WORKLOADS[name]
    B = Bg if B is None else B
    layers = make_layers(name, seed)
    op = IAFOperator(variant, n_z, hidden, [n_z, n_z], nl="elu", path="auto")
    op.set_weights([tuple(t.to(device) for t in l) for l in layers])
    g = torch.Generator().manual_seed(seed)
    sets = []
    logdets = torch.zeros((nsets, B), device=device)  # one row per set: an ELBO scalar is one .sum() over E rows
    for i in range(nsets):
        z = torch.randn((B, n_z, H, W), generator=g)
        ctx = 0.1 * torch.randn((B, hidden[0], H, W), generator=g)
        sets.append(dict(z=z.to(device), ctx=ctx.to(device), z_out=torch.empty((B, n_z, H, W), device=device),
                         logsd=torch.empty((B, n_z, H, W), device=device), logdet=logdets[i]))
    op.logdets = logdets
    return op, layers, sets


# ----------------------------------------------------------------------------------------------
# the CPU arm (used by --impl reference directly and, through a subprocess, by the b200 arm)
# ----------------------------------------------------------------------------------------------
def cpu_port_runner(name, layers_cpu, sample_B):
    """Returns (fn, elems_per_call): one reference-path IAF step on the host cores."""
    from oracle import iaf_oracle_torch as OT
    variant, n_z, hidden, H, W, B, E = WORKLOADS[name]
    g = torch.Generator().manual_seed(0)
    z = torch.randn((sample_B, n_z, H, W), generator=g)
    ctx = 0.1 * torch.randn((sample_B, hidden[0], H, W), generator=g)
    keys = ("V", "g", "b") if variant == "tf" else ("w", "s", "b")
    hid = [dict(zip(keys, l)) for l in layers_cpu[:len(hidden)]]
    heads = [dict(zip(keys, l)) for l in layers_cpu[len(hidden):]]

    def fn():
        with torch.no_grad():
            return OT.iaf_step(variant, z, ctx, hid, heads, "elu")
    return fn, sample_B * n_z * H * W


def _timed_calls(fn, warmup, n):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(n):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return ts


def cpu_arm(name, steps, warmup):
    """The reference's CPU path on this box: returns (seconds per step [median], info dict).  Thread count: the
    frameworks of the reference pick their own; torch gets slower past what these conv sizes can use, so every candidate
    (8, 16, the physical cores of one NUMA node, all physical cores) gets 3 warm-up + 5 timed calls and the best median
    runs the measurement proper (``warmup`` + ``steps`` calls of the full 256-sample batch, median)."""
    variant, n_z, hidden, H, W, B, E = WORKLOADS[name]
    allowed, n_phys, n_node = host_topology()
    layers = make_layers(name)
    fn, elems = cpu_port_runner(name, layers, B)
    cands = sorted({c for c in (8, 16, n_node, n_phys) if 1 <= c <= len(allowed)}) or [len(allowed)]
    cand_ms = {}
    for c in cands:
        torch.set_num_threads(c)
        cand_ms[c] = statistics.median(_timed_calls(fn, 3, 5)) * 1e3
    best = min(cand_ms, key=cand_ms.get)
    torch.set_num_threads(best)
    # at least 20 timed calls whatever K is: single calls on a shared host scatter by an order of magnitude (10 ms median,
    # 170 ms maximum seen on the GPU boxes), and the two arms must report the same number for the same routine
    steps = max(20, min(steps, 50))
    warmup = max(5, min(warmup, 10))
    ts = _timed_calls(fn, warmup, steps)
    t = statistics.median(ts)
    info = {"value": elems / t, "unit": UNIT, "cores": best, "kind": "port",
            "sample": "the full %d-sample batch per step, %d warm-up + %d timed steps (median step %.2f ms, min %.2f, "
                      "max %.2f), torch-CPU fp32 port of the reference path (Theano/TF originals cannot run here)" % (
                          B, warmup, steps, t * 1e3, min(ts) * 1e3, max(ts) * 1e3),
            "candidates_ms": {str(k): round(v, 3) for k, v in cand_ms.items()},
            "host": {"allowed_cpus": len(allowed), "physical_cores": n_phys, "physical_cores_per_numa_node": n_node},
            "steps": steps, "warmup": warmup}
    return t, info


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU path (torch-CPU port of the oracle), rank 0 only."""
    if rank != 0:
        return
    name = args.workload
    variant, n_z, hidden, H, W, B, E = WORKLOADS[name]
    t, info = cpu_arm(name, args.steps, args.warmup)
    value = info["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": info["steps"],
        "warmup": info["warmup"], "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(name), "global_batch": B, "timing": "median step, host clock"},
        "cpu_baseline": info,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def cpu_baseline_subprocess(name, steps, warmup, full_affinity):
    """The b200 arm's cpu_baseline leg: the SAME routine, in a fresh process with the original CPU affinity (this process
    is bound to the GPU's NUMA node and carries a CUDA context, an NVML poller and pinned buffers)."""
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "CUDA_VISIBLE_DEVICES")}
    env["CUDA_VISIBLE_DEVICES"] = ""

    def unbind():
        try:
            os.sched_setaffinity(0, full_affinity)
        except Exception:
            pass
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", name,
                            "--steps", str(steps), "--warmup", str(warmup)], env=env, preexec_fn=unbind,
                           capture_output=True, text=True, timeout=600)
        line = json.loads(r.stdout.strip().splitlines()[-1])
        return line["cpu_baseline"]
    except Exception as e:  # pragma: no cover
        return {"value": None, "unit": UNIT, "cores": None, "kind": "port", "sample": "failed: %r" % (e,)}


# ----------------------------------------------------------------------------------------------
# device-side measurement of one workload
# ----------------------------------------------------------------------------------------------
class DeviceBench(object):
    def __init__(self, name, device, world, rank, dist, use_graph=True):
        import ctypes as C
        self.C = C
        self.name, self.device, self.world, self.rank, self.dist, self.use_graph = name, device, world, rank, dist, use_graph
        variant, n_z, hidden, H, W, Bg, E = WORKLOADS[name]
        if Bg % world != 0:
            raise SystemExit("global batch %d does not divide over %d ranks" % (Bg, world))
        self.B = Bg // world
        self.Bg, self.n_z, self.hidden, self.H, self.W, self.E = Bg, n_z, hidden, H, W, E
        self.alg_bytes_unit = 4 * self.B * H * W * (n_z + hidden[0] + n_z + n_z) + 4 * self.B
        nsets = max(2, -(-3 * 126 * 2 ** 20 // self.alg_bytes_unit))  # footprint >= 3x the 126 MB L2
        self.nsets = -(-nsets // E) * E                                # a whole number of ELBO groups
        self.op, self.layers_cpu, self.sets = make_workload(name, device, self.nsets, B=self.B)
        self.lib = self.op._lib
        self.plan = self.op._plan(H, W, device)
        self.stream = torch.cuda.current_stream(device)
        self.side = torch.cuda.Stream(device)

    def launch(self, i, st):
        C = self.C
        s = self.sets[i % self.nsets]
        rc = self.lib.iaf_step_fwd(self.plan, C.c_void_p(s["z"].data_ptr()), C.c_void_p(s["ctx"].data_ptr()),
                                   C.c_void_p(s["z_out"].data_ptr()), C.c_void_p(s["logsd"].data_ptr()),
                                   C.c_void_p(s["logdet"].data_ptr()), self.B, C.c_void_p(st.cuda_stream))
        if rc != 0:
            from iaf_b200 import _lib
            _lib.check(rc)

    def _capture(self, idxs, tail=None):
        """One CUDA graph launching steps ``idxs`` back to back (then ``tail()``, e.g. the group's scalar reduction);
        None when --no-graph or capture is unsupported."""
        if not self.use_graph:
            return None
        try:
            gstream = torch.cuda.Stream(self.device)
            gstream.wait_stream(self.stream)
            with torch.cuda.stream(gstream):
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, stream=gstream):
                    for i in idxs:
                        self.launch(i, torch.cuda.current_stream(self.device))
                    if tail is not None:
                        tail()
            self.stream.wait_stream(gstream)
            return graph
        except Exception as e:  # capture unsupported -> direct launches (still the CUDA path)
            self.capture_error = type(e).__name__
            torch.cuda.synchronize()
            return None

    def warmup(self, Wm):
        lc0 = self.op.launch_count()
        for i in range(Wm):
            self.launch(i, self.stream)
        torch.cuda.synchronize()
        self.launches_per_step = (self.op.launch_count() - lc0) // Wm  # 1 (fused / SIMT) or one per conv stage (layered)

    def _barrier(self):
        torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()
            torch.cuda.synchronize()

    def _max_over_ranks(self, vals):
        tt = torch.tensor(vals, device=self.device, dtype=torch.float64)
        if self.dist is not None:
            self.dist.all_reduce(tt, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in tt]

    def time_kernels(self, K):
        """Kernel-only region: K back-to-back launches (one graph), CUDA events on the launching stream."""
        g = self._capture(range(K))
        if g is not None:
            g.replay()
        self._barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if g is not None:
            g.replay()
        else:
            for i in range(K):
                self.launch(i, self.stream)
        e1.record()
        self._barrier()
        (ms,) = self._max_over_ranks([e0.elapsed_time(e1)])
        self.launch_mode = "cuda_graph" if g is not None else "direct"
        return ms * 1e-3 / K

    def time_elbo_groups(self, K):
        """The job as the model runs it: groups of E steps, each followed by the ELBO scalar (sum of the group's
        log-dets) and one all-reduce of it across ranks on a side stream.  Returns (seconds per step, launches, scalar)."""
        E, nsets = self.E, self.nsets
        groups = [(s, min(E, K - s)) for s in range(0, K, E)]
        scal = torch.zeros((len(groups),), device=self.device)
        rows = self.op.logdets

        def reduce_group(gi, s, n):  # the ELBO term of this evaluation on this rank's shard
            r0 = s % nsets
            torch.sum(rows[r0:r0 + n].reshape(-1), dim=0, out=scal[gi])
        reduce_group(0, 0, groups[0][1])  # outside any capture first (lazy initialisation of the reduction)
        # one graph per ELBO evaluation: its E step launches and the reduction of their log-dets into scal[gi]
        # one rank: nothing happens between two evaluations (no collective), so the K steps and their reductions are ONE graph
        whole = None
        if self.dist is None and self.use_graph:
            def all_groups():
                for gi, (s, n) in enumerate(groups):
                    for i in range(s, s + n):
                        self.launch(i, torch.cuda.current_stream(self.device))
                    reduce_group(gi, s, n)
            whole = self._capture([], tail=all_groups)
        graphs = [None] * len(groups)
        if whole is None:
            graphs = [self._capture(range(s, s + n), tail=(lambda gi=gi, s=s, n=n: reduce_group(gi, s, n)))
                      for gi, (s, n) in enumerate(groups)]

        def run():
            if whole is not None:
                whole.replay()
                return
            works = []
            for gi, (s, n) in enumerate(groups):
                g = graphs[gi]
                if g is not None:
                    g.replay()
                else:
                    for i in range(s, s + n):
                        self.launch(i, self.stream)
                    reduce_group(gi, s, n)
                if self.dist is not None:
                    self.side.wait_stream(self.stream)
                    with torch.cuda.stream(self.side):
                        works.append(self.dist.all_reduce(scal[gi], async_op=True))  # tf_train.py:142, one per ELBO
            if works:
                with torch.cuda.stream(self.side):
                    for w in works:
                        w.wait()
                self.stream.wait_stream(self.side)
        run()  # one untimed pass (warms the reduction, the collective and the graphs)
        self._barrier()
        l0 = self.op.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run()
        e1.record()
        self._barrier()
        (ms,) = self._max_over_ranks([e0.elapsed_time(e1)])
        direct = self.op.launch_count() - l0
        n_launched = direct if direct else K * self.launches_per_step  # graph replays do not pass through the C ABI
        self.elbo_scalars = scal
        return ms * 1e-3 / K, int(n_launched), float(scal.sum()), len(groups)

    def last_step_outputs(self, K):
        """What a caller of the timed path holds after its last step (step K-1): z', arw_logsd and the per-sample logdet of
        that step, and the ELBO scalar of the evaluation the step closed.  At N > 1 the shards are gathered over ranks
        (a collective: every rank calls this)."""
        s = self.sets[(K - 1) % self.nsets]
        out = {"z_out": s["z_out"], "logsd": s["logsd"], "logdet": s["logdet"]}
        if self.dist is not None:
            for k, v in out.items():
                full = torch.empty((self.world * v.shape[0],) + tuple(v.shape[1:]), device=self.device, dtype=v.dtype)
                self.dist.all_gather_into_tensor(full, v.contiguous())
                out[k] = full
        out["elbo_logdet_sum"] = self.elbo_scalars[-1:]
        return {k: v.cpu().numpy() for k, v in out.items()}

    def training_pair(self, iters=20):
        """Forward that keeps the activations (iaf_step_fwd_train) and backward from them (iaf_step_bwd_saved: gradients of z,
        context and every parameter), the pair the autograd node of IAFOperator.step runs; CUDA events, this rank's shard."""
        op, s = self.op, self.sets[0]
        z, ctx = s["z"], s["ctx"]
        g1 = torch.randn_like(z)
        gl = torch.randn(self.B, device=self.device)

        def timed(fn):
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / iters * 1e3
        t_f = timed(lambda: op._step_train_raw(z, ctx))
        zo, ls, _, hs = op._step_train_raw(z, ctx)
        t_b = timed(lambda: op._backward("step", z, ctx, op._layers, (g1, g1, gl), True, saved=(zo, ls, hs)))
        return {"fwd_train_us": t_f, "bwd_saved_us": t_b, "samples": self.B,
                "backward_path": op.backward_path(self.H, self.W, self.device)}

    def roofline(self, t_kernel):
        hbm_gbs, bf16_tf, peak_src = measured_peaks()
        op, H, W, dev = self.op, self.H, self.W, self.device
        alg_bytes = op.algorithmic_bytes(self.B, H, W, dev)
        alg_flops = op.algorithmic_flops(self.B, H, W, dev)
        t_hbm, t_tc = alg_bytes / (hbm_gbs * 1e9), alg_flops / (bf16_tf * 1e12)
        if t_hbm >= t_tc:
            achieved = alg_bytes / t_kernel / 1e9
            roof = {"bound": "hbm", "achieved": achieved, "peak": hbm_gbs, "unit": "GB/s", "frac": achieved / hbm_gbs}
        else:
            achieved = alg_flops / t_kernel / 1e12
            roof = {"bound": "tensor", "achieved": achieved, "peak": bf16_tf, "unit": "TFLOP/s", "frac": achieved / bf16_tf}
        roof.update({"traffic": None, "kernel": "iaf_step (%s path, %d launch%s per step)" % (
                         op.path_used(H, W, dev), self.launches_per_step, "" if self.launches_per_step == 1 else "es"),
                     "kernel_us": t_kernel * 1e6, "algorithmic_bytes": alg_bytes, "algorithmic_flops": alg_flops,
                     "floor_us": {"hbm": t_hbm * 1e6, "tensor": t_tc * 1e6}, "samples_per_launch": self.B,
                     "peak_source": peak_src})
        return roof

    def time_e2e(self, K):
        """Host buffers through the public API: every step pinned host inputs -> H2D -> step -> D2H of z', arw_logsd,
        logdet into pinned host outputs (iaf_step_submit_host: three staging slots, so copy-in of step i+1, the kernel of
        step i and copy-out of step i-1 overlap); the region ends after wait_host().  At least 100 steps and 0.5 s."""
        op, B, n_z, H, W, hidden, nsets = self.op, self.B, self.n_z, self.H, self.W, self.hidden, self.nsets
        NH = 4
        hz = [torch.empty((B, n_z, H, W)).pin_memory().copy_(self.sets[i % nsets]["z"].cpu()) for i in range(NH)]
        hc = [torch.empty((B, hidden[0], H, W)).pin_memory().copy_(self.sets[i % nsets]["ctx"].cpu()) for i in range(NH)]
        ho = [torch.empty((B, n_z, H, W)).pin_memory() for _ in range(NH)]
        hl = [torch.empty((B, n_z, H, W)).pin_memory() for _ in range(NH)]
        hd = [torch.empty((B,)).pin_memory() for _ in range(NH)]

        def run(n):
            t0 = time.perf_counter()
            for i in range(n):
                op.submit_host(hz[i % NH], hc[i % NH], ho[i % NH], hl[i % NH], hd[i % NH])
            op.wait_host()
            return time.perf_counter() - t0
        run(8)
        Ke = max(K, 100)
        self._barrier()
        t = run(Ke)
        if t < 0.5:  # too short a window for a host-clock measurement: size it to ~0.6 s and measure again
            Ke = int(Ke * 0.6 / max(t, 1e-4)) + 1
            (kmax,) = self._max_over_ranks([float(Ke)])
            Ke = int(kmax)
            self._barrier()
            t = run(Ke)
        check = float(hd[(Ke - 1) % NH].sum())  # the step's result is read on the host
        (t,) = self._max_over_ranks([t])
        h2d = hz[0].numel() * 4 + hc[0].numel() * 4
        d2h = ho[0].numel() * 4 + hl[0].numel() * 4 + hd[0].numel() * 4
        return t / Ke, Ke, h2d, d2h, check


DUMP_LIMIT_BYTES = 64 * 2 ** 20


def dump_outputs(d, outs):
    """Writes ``outs`` as d/<name>.npy.  Arrays with a leading batch axis that together exceed DUMP_LIMIT_BYTES keep a fixed,
    seeded sample of their rows (the same rows for the same batch size), in ascending order."""
    batched = [k for k in outs if k != "elbo_logdet_sum"]
    nb = outs[batched[0]].shape[0]
    per_row = sum(outs[k].nbytes for k in batched) // nb
    keep = min(nb, DUMP_LIMIT_BYTES // per_row)
    if keep < nb:
        rows = np.sort(np.random.RandomState(0).choice(nb, keep, replace=False))
        outs = dict(outs, **{k: outs[k][rows] for k in batched})
    os.makedirs(d, exist_ok=True)
    for k, v in outs.items():
        np.save(os.path.join(d, k + ".npy"), np.ascontiguousarray(v, dtype=np.float32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2a", choices=sorted(WORKLOADS))  # c2a = the headline
    ap.add_argument("--no-graph", action="store_true", help="direct launches instead of CUDA graphs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="skip the second headline shape")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--batch", type=int, default=0, help="development: override the workload's global batch")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's outputs as DIR/<name>.npy (float32, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the b200 arm computed")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    full_affinity = set(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else None
    binding = bind_to_gpu_numa(local_rank)  # before the CUDA context and any pinned allocation
    import __graft_entry__
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    if rank == 0:
        __graft_entry__.build()
    if dist is not None:
        dist.barrier()

    name = args.workload
    if args.batch:
        WORKLOADS[name] = WORKLOADS[name][:5] + (args.batch,) + WORKLOADS[name][6:]
    K, Wm = args.steps, args.warmup
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        sampler.phase = "warmup"
    db = DeviceBench(name, device, world, rank, dist, use_graph=not args.no_graph)
    db.warmup(Wm)
    if sampler:
        sampler.phase = "timed"
    t_kernel = db.time_kernels(K)
    t_step, n_launched, elbo_sum, n_groups = db.time_elbo_groups(K)
    outs = db.last_step_outputs(K) if args.dump_outputs else None
    if sampler:
        sampler.phase = "between"
    elems_step = db.Bg * db.n_z * db.H * db.W
    value = elems_step / t_step
    roof = db.roofline(t_kernel)

    e2e = None
    if not args.no_e2e:
        if sampler:
            sampler.phase = "e2e"
        t_e2e, Ke, h2d, d2h, check = db.time_e2e(K)
        e2e = {"value": elems_step / t_e2e, "unit": UNIT, "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h * world,
               "ms_per_step": t_e2e * 1e3, "steps": Ke, "logdet_sum_last_step": check, "host_binding": binding,
               "entry": "IAFOperator.submit_host/wait_host -> iaf_step_submit_host (3-slot H2D/compute/D2H pipeline), "
                        "every rank its shard of the global batch"}
        if sampler:
            sampler.phase = "between"

    # ---- the other headline shape, device-timed in the same run ----
    also = None
    if not args.no_also and name == "c2a":
        other = "c2b"
        if sampler:
            sampler.phase = "timed"
        ob = DeviceBench(other, device, world, rank, dist, use_graph=not args.no_graph)
        ob.warmup(max(3, Wm // 2))
        Ko = max(20, min(K, 100))
        ot_kernel = ob.time_kernels(Ko)
        ot_step, on_launched, _, o_groups = ob.time_elbo_groups(Ko)
        o_elems = ob.Bg * ob.n_z * ob.H * ob.W
        also = {("c2b" if world == 1 else "c5"): {
            "workload": workload_string(other) + (" (C5: sharded %d/GPU)" % ob.B if world > 1 else ""),
            "value": o_elems / ot_step, "unit": UNIT, "steps": Ko, "ms_per_step": ot_step * 1e3,
            "steps_per_elbo": ob.E, "elbo_evaluations": o_groups, "gpu_launches": on_launched,
            "kernels_per_step": ob.launches_per_step, "roofline": ob.roofline(ot_kernel)}}
        if world == 1:  # the training pair of both headline shapes (SURVEY 8f-4), device-timed in the same run
            also["training_pair"] = {"c2a": db.training_pair(), "c2b": ob.training_pair(10)}
        if sampler:
            sampler.phase = "between"
        del ob
    clocks = sampler.finish() if sampler else None

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    cpu = None
    if not args.no_cpu_baseline and world == 1:
        cpu = cpu_baseline_subprocess(name, 20, 3, full_affinity)

    path = db.op.path_used(db.H, db.W, device)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": t_step * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32 (tc path: fp16 hi/lo operand pairs, three products per MAC, f32 accumulate)" if path == "tc" else "f32",
        "data": "synthetic",
        "config": {"workload": workload_string(name), "global_batch": db.Bg, "samples_per_gpu": db.B,
                   "parallelism": "dp%d" % world, "path": path, "launch": db.launch_mode,
                   "kernels_per_step": db.launches_per_step, "steps_per_elbo": db.E, "elbo_evaluations": n_groups,
                   "l2": "rotating %d input/output sets (%.0f MB > 126 MB L2)" % (db.nsets, db.nsets * db.alg_bytes_unit / 2 ** 20),
                   "collective": ("one NCCL all-reduce of the ELBO scalar per evaluation (%d steps), on a side stream"
                                  % db.E) if world > 1 else "none",
                   "samples_per_s": value / (db.n_z * db.H * db.W)},
        "e2e": e2e,
        "gpu_launches": int(n_launched),
        "clocks": clocks,
        "roofline": roof,
        "cpu_baseline": cpu,
        "also": also,
        "elbo_scalar": elbo_sum,
    }
    if outs is not None:
        dump_outputs(args.dump_outputs, outs)
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
