"""Time to collision in isolation: tds_time_to_collision forward and backward at config 2 (1024 envs x 64 agents on
carla_Town01, at road positions as bench.py seeds them) and at config 4's agent count (64 envs x 512 agents, uniform
in a 120 m square, speeds U[0, 15] m/s), each at a horizon of 3 s and 8 s.  Beside them the eager torch statement of
the definition over all pairs (tests/test_gpu_time_to_collision.ttc_ref, one op per operation).  The kernels are timed
with CUDA events around CUDA-graph replays after warm-up (profiles/time_observations.graph_us); the eager statement,
which synchronises on the host, with CUDA events around eager calls.  The kernels read 26 bytes per agent and write
12 bytes per origin.  Prints one JSON line per case and a final line with the card name and power limit.

  python profiles/time_time_to_collision.py [--reps 20]
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

HORIZONS = (3.0, 8.0)


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


def inputs(name, dev):
    """(state [B,N,4], size [B,N,2], present [B,N]) of a case."""
    import bench
    if name == "config2_1024x64":
        state, size, _, _ = bench.synth_inputs(1024, 64, 1000, 1)
    else:
        rng = np.random.default_rng(1000)
        B, N = 64, 512
        state = np.concatenate([rng.uniform(0, 120, (B, N, 2)), rng.uniform(-np.pi, np.pi, (B, N, 1)),
                                rng.uniform(0, 15, (B, N, 1))], -1).astype(np.float32)
        size = np.tile(np.array(bench.VEH[:2], np.float32), (B, N, 1))
    state, size = torch.tensor(state, device=dev), torch.tensor(size, device=dev)
    return state, size, torch.ones(state.shape[:2], dtype=torch.bool, device=dev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    from torchdrivesim_b200 import ops
    from tests.test_gpu_time_to_collision import ttc_ref
    dev = torch.device("cuda")
    res = {"card": card(), "reps": args.reps}
    gen = torch.Generator(device=dev).manual_seed(0)
    for name in ("config2_1024x64", "config4_64x512"):
        state, size, present = inputs(name, dev)
        B, N = present.shape
        for H in HORIZONS:
            ttc, idx = ops._time_to_collision_fwd(state, size, present, None, H)
            grad = torch.randn(B, N, device=dev, generator=gen)
            entry = {"envs": B, "agents": N, "pairs": B * N * (N - 1), "horizon_s": H,
                     "contact": round(float((idx >= 0).float().mean()), 4),
                     "contact_at_0": round(float((ttc == 0).float().mean()), 4)}
            entry["fwd_us"] = round(graph_us(lambda c: ops._time_to_collision_fwd(state, size, present, None, H), 1, 4,
                                             args.reps), 2)
            entry["bwd_us"] = round(graph_us(lambda c: ops._time_to_collision_bwd(state, size, present, None, H, idx,
                                                                                   grad), 1, 4, args.reps), 2)
            entry["eager_torch_fwd_us"] = round(1e3 * eager_ms(lambda: ttc_ref(state, size, present, N, H), 2), 1)
            entry["speedup_fwd"] = round(entry["eager_torch_fwd_us"] / entry["fwd_us"], 1)
            key = f"{name}_H{H:g}s"
            res[key] = entry
            print(json.dumps({key: entry}), flush=True)
            del ttc, idx, grad
            torch.cuda.empty_cache()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
