"""Range-scan observations in isolation: tds_range_scan forward and backward at config 2 (1024 envs x 64 agents on
carla_Town01, at road positions as bench.py seeds them), R = 32 / 64 / 256 rays, max_range 30 m and 50 m, with and
without the lane markings, and at 64 envs x 512 agents (agents only, 50 m).  Beside them the eager torch brute force of
the definition (tests/test_gpu_range_scan.scan_ref: every box edge and every marking within reach of every origin,
chunked over origins), and, as context only, the raster kernel of a 64x64 birdview step at config 2 (the observation a
range scan can stand in for).  The kernels are timed with CUDA events around CUDA-graph replays after warm-up
(profiles/time_observations.graph_us); the brute force and the raster, which synchronise on the host, with CUDA events
around eager calls.  The kernels read 24 bytes per agent and the map's segment grid (~160 KB), which stays in L2.
Prints one JSON line per case and a final line with the card name and power limit.

  python profiles/time_range_scan.py [--reps 20]
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from time_offroad import card  # noqa: E402
from time_observations import graph_us  # noqa: E402

RAYS = (32, 64, 256)
RANGES = (30.0, 50.0)


def eager_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def raster_ms(B, A, dev):
    """The raster kernel alone at B x A cameras, 64x64 (CUDA events the library records around its launch)."""
    import bench
    import torchdrivesim_b200 as tds
    state, size, lr, _ = bench.synth_inputs(B, A, 1000, 1)
    km = tds.KinematicBicycle(left_handed=True)
    km.set_params(lr=torch.tensor(lr, device=dev))
    km.set_state(torch.tensor(state, device=dev))
    sim = tds.Simulator(tds.StaticMap.from_npz(bench.map_npz()), km, torch.tensor(size, device=dev),
                        torch.ones(B, A, dtype=torch.bool, device=dev), tds.TorchDriveConfig(left_handed_coordinates=True))
    out = torch.empty(B, A, 3, bench.RES, bench.RES, device=dev)
    for _ in range(3):
        sim.render_egocentric(out=out)
    lib = tds._lib.load()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(10)]
    for a, b in evs:
        lib.tds_raster_set_timing_events(a.cuda_event, b.cuda_event)
        sim.render_egocentric(out=out)
    lib.tds_raster_set_timing_events(None, None)
    torch.cuda.synchronize()
    return float(np.median([a.elapsed_time(b) for a, b in evs]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    import bench
    import torchdrivesim_b200 as tds
    from torchdrivesim_b200 import ops
    from tests.test_gpu_range_scan import scan_ref
    dev = torch.device("cuda")
    town = tds.StaticMap.from_npz(bench.map_npz())
    res = {"card": card(), "reps": args.reps}
    gen = torch.Generator(device=dev).manual_seed(0)
    cases = [("config2_1024x64", 1024, 64, R, md, mk) for R in RAYS for md in RANGES for mk in (True, False)]
    cases += [("whole_64x512", 64, 512, R, 50.0, False) for R in RAYS]
    inputs = {}
    for name, B, A, R, md, markings in cases:
        if (B, A) not in inputs:
            state, size, _, _ = bench.synth_inputs(B, A, 1000, 1)
            inputs[(B, A)] = torch.tensor(np.concatenate([state[..., :3], size, np.ones_like(size[..., :1])], -1), device=dev)
        absolute = inputs[(B, A)]
        ms = tds.MapSet([town]) if markings else None
        grad = torch.randn(B, A, R, device=dev, generator=gen)
        dist, kind, idx = ops._range_scan_fwd(absolute, R, None, md, ms)
        entry = {"agents": B * A, "rays": R, "max_range": md, "markings": markings,
                 "hit_agent": round(float((kind == 0).float().mean()), 4),
                 "hit_marking": round(float((kind == 1).float().mean()), 4)}
        entry["fwd_us"] = round(graph_us(lambda c: ops._range_scan_fwd(absolute, R, None, md, ms), 1, 4, args.reps), 2)
        entry["bwd_us"] = round(graph_us(lambda c: ops._range_scan_bwd(absolute, R, None, ms, kind, idx, grad), 1, 4,
                                         args.reps), 2)
        chunk = max(64, int(3e8 // (R * (4 * A + 1500))))         # origins per brute-force chunk: ~1.2 GB per tensor
        entry["brute_force_fwd_us"] = round(1e3 * eager_ms(lambda: scan_ref(absolute, R, A, md, ms, chunk=chunk), 2), 1)
        entry["speedup_fwd"] = round(entry["brute_force_fwd_us"] / entry["fwd_us"], 1)
        key = f"{name}_R{R}_{md:g}m_{'markings' if markings else 'agents'}"
        res[key] = entry
        print(json.dumps({key: entry}), flush=True)
        del grad, dist, kind, idx
        torch.cuda.empty_cache()
    res["raster_config2_ms"] = round(raster_ms(bench.ENVS_PER_GPU, bench.AGENTS, dev), 3)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
