"""Time one data-dependent initialisation call (IAFOperator.data_init -> iaf_multiconv_init) on one GPU: CUDA events
around each call, inputs resident in HBM, after two warm-up calls.  The pass runs once per training run, so the number
records its cost; no target is set.  One call = re-pack + per stage (conv, statistics, parameters, output) on the
exact-fp32 kernels, whatever the plan's path.  Prints one JSON line per workload with the device name and power limit.
usage: python tools/bench_init.py [calls]"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from iaf_b200 import IAFOperator  # noqa: E402
from oracle import iaf_oracle as O  # noqa: E402  (synthetic parameter / input generator only)

WL = {"c2a": [64], "c2b": [160, 160]}


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # the number still stands; say why the limit is missing
        return "unavailable (%s)" % e


def main():
    calls = int(sys.argv[1]) if len(sys.argv) > 1 else 10
    n_z, H, W = 32, 16, 16
    device = {"name": torch.cuda.get_device_name(0), "power_limit,max_sm_clock": power_limit()}
    for wl, hidden in WL.items():
        hid, hd = O.make_params("tf", n_z, hidden, [n_z, n_z], seed=1)
        for B in (16, 256):
            z, ctx = O.make_inputs(B, n_z, hidden[0], H, W, seed=0)
            dev = [tuple(torch.from_numpy(np.ascontiguousarray(l[k])).cuda() for k in "Vgb") for l in hid + hd]
            op = IAFOperator("tf", n_z, hidden, [n_z, n_z], nl="elu").set_weights(dev)
            zg, cg = torch.from_numpy(z).cuda(), torch.from_numpy(ctx).cuda()
            for _ in range(2):
                op.data_init(zg, cg)
            torch.cuda.synchronize()
            l0 = op.launch_count()
            ms = []
            for _ in range(calls):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                op.data_init(zg, cg)
                e1.record()
                torch.cuda.synchronize()
                ms.append(e0.elapsed_time(e1))
            print(json.dumps({"workload": wl, "B": B, "H": H, "W": W, "path": op.path_used(H, W, "cuda:0"),
                              "data_init_ms_median": float(np.median(ms)), "data_init_ms_min": float(np.min(ms)),
                              "data_init_ms_max": float(np.max(ms)), "calls": calls,
                              "launches_per_call": (op.launch_count() - l0) // calls, "device": device}), flush=True)


if __name__ == "__main__":
    main()
