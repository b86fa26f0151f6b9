"""Offroad forward in isolation, CUDA events: the benchmark's 1024 x 64 agents on carla_Town01, threshold 0.5, with the
corner triage on and off (TDS_OFFROAD_TRIAGE=0), agents on road vertices and displaced by N(0, 3 m) / N(0, 10 m).  Also
times tds_infraction_metrics at the same size.  Prints one JSON line (with the card name and power limit).

  python profiles/time_offroad.py [--iters 200]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True).strip()
    except (OSError, subprocess.CalledProcessError):
        return torch.cuda.get_device_name()


def time_ms(fn, iters):
    for _ in range(10):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    args = ap.parse_args()
    import bench
    import torchdrivesim_b200 as tds
    dev = torch.device("cuda")
    B, A = bench.ENVS_PER_GPU, bench.AGENTS
    state, size, _, _ = bench.synth_inputs(B, A, 1000, 1)
    town = tds.MapSet([tds.StaticMap.from_npz(bench.map_npz())])
    rng = np.random.default_rng(0)
    out = torch.empty(B, A, device=dev)
    res = {"card": card(), "agents": B * A, "threshold": 0.5, "iters": args.iters, "offroad_fwd_us": {}}
    for displace in (0.0, 3.0, 10.0):
        st = state.copy()
        st[..., :2] += (displace * rng.standard_normal((B, A, 2))).astype(np.float32)
        st_d, sz_d = torch.tensor(st, device=dev), torch.tensor(size, device=dev)
        for triage in ("1", "0"):
            os.environ["TDS_OFFROAD_TRIAGE"] = triage
            ms = time_ms(lambda: tds.ops.offroad(st_d, sz_d, town, 0.5, out=out), args.iters)
            res["offroad_fwd_us"][f"displace_{displace:g}m_triage_{'on' if triage == '1' else 'off'}"] = round(ms * 1e3, 2)
    os.environ.pop("TDS_OFFROAD_TRIAGE")
    coll = torch.rand(B, A, device=dev)
    acc = torch.zeros(6, dtype=torch.float64, device=dev)
    res["infraction_metrics_us"] = round(time_ms(lambda: tds.ops.infraction_metrics(coll, out, None, acc), args.iters) * 1e3, 2)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
