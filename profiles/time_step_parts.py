"""The launches of the benchmark's graphed step (bench.py: 1024 environments x 64 agents, carla_Town01, 64x64 birdviews,
discs collisions + offroad), one by one.

  python profiles/time_step_parts.py [--tree DIR] [--steps 200]

* step_ms: CUDA events around replays of GraphedHotPath (the bench step without its infraction metrics), blocks of 8
  steps from the benchmark's initial state;
* kernels_us / timeline_us: mean device time of every kernel of a replay, and its mean start and end relative to the
  start of the step's kinematic kernel, from torch.profiler (CUPTI) over 8 replays after the timed ones;
* allpairs_us: the discs all-pairs kernel alone at the benchmark's boxes and at config 3's shape (512 x 128), and the IoU
  kernel at config 4's (64 x 512), CUDA events around replays of a CUDA graph of 20 launches each.

--tree times the package of another checkout (e.g. the parent commit's, for a before / after comparison) with this
script.  Prints one JSON line with the card's name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True).strip()
    except (OSError, subprocess.CalledProcessError):
        return torch.cuda.get_device_name()


def graph_us(fn, launches=20, replays=50):
    """Mean µs of one fn() when `launches` of them are replayed as one CUDA graph."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        for _ in range(launches):
            fn()
    for _ in range(5):
        g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(replays):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / (replays * launches)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tree", default=ROOT)
    ap.add_argument("--steps", type=int, default=200)
    args = ap.parse_args()
    tree = os.path.abspath(args.tree)
    sys.path.insert(0, tree)
    import bench
    import torchdrivesim_b200 as tds
    assert os.path.dirname(os.path.dirname(os.path.abspath(tds.__file__))) == tree, tds.__file__
    dev = torch.device("cuda:0")
    B, A = bench.ENVS_PER_GPU, bench.AGENTS
    state, size, lr, actions = bench.synth_inputs(B, A, 1000, 8)
    town = tds.StaticMap.from_npz(bench.map_npz())
    km = tds.KinematicBicycle(left_handed=True)
    km.set_params(lr=torch.tensor(lr, device=dev))
    km.set_state(torch.tensor(state, device=dev))
    sim = tds.Simulator(town, km, torch.tensor(size, device=dev), torch.ones(B, A, dtype=torch.bool, device=dev),
                        tds.TorchDriveConfig(left_handed_coordinates=True))
    act = torch.tensor(actions, device=dev)
    runner = tds.GraphedHotPath(sim, render=True)
    res = {"card": card(), "tree": "this tree" if tree == ROOT else f"--tree {os.path.basename(tree)}", "workload": f"bench.py step, {B} x {A}, {bench.RES}x{bench.RES}"}

    # the agents drive off the road (and, after a few hundred steps, off the map) under random actions: every block of 8
    # timed steps starts from the benchmark's initial state again, as bench.py's timed steps do
    state0 = torch.tensor(state, device=dev)
    for i in range(24):
        if i % 8 == 0:
            runner.set_state(state0)
        runner.run(act[i % 8])
    torch.cuda.synchronize()
    total = 0.0
    blocks = max(args.steps // 8, 1)
    for _ in range(blocks):
        runner.set_state(state0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(8):
            runner.run(act[i])
        e1.record()
        torch.cuda.synchronize()
        total += e0.elapsed_time(e1)
    res["step_ms"] = total / (8 * blocks)

    from torch.profiler import ProfilerActivity, profile
    n = 8
    runner.set_state(state0)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(n):
            runner.run(act[i])
        torch.cuda.synchronize()
    launches = []
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA and "Memcpy" not in ev.name and "Memset" not in ev.name:
            name = ev.name.replace("(anonymous namespace)::", "")
            if name.endswith(")"):                  # drop the parameter list
                depth, k = 0, len(name) - 1
                while k >= 0:
                    depth += name[k] == ")"
                    depth -= name[k] == "("
                    if depth == 0:
                        break
                    k -= 1
                name = name[:k]
            launches.append((ev.time_range.start, ev.time_range.end, name[:100]))
    # the timeline of a step: every launch's start and end relative to the start of the step's kin_fwd_kernel (a name
    # met twice in a step gets " #2"); kernels of the collision / offroad branch run beside the raster's, so their
    # durations overlap rather than add up
    kernels, timeline, step = {}, {}, None
    for t0, t1, name in sorted(launches):
        if name.endswith("kin_fwd_kernel"):
            step, seen = t0, {}
        if step is None:
            continue
        seen[name] = seen.get(name, 0) + 1
        key = name if seen[name] == 1 else f"{name} #{seen[name]}"
        kernels.setdefault(key, []).append(t1 - t0)
        timeline.setdefault(key, []).append((t0 - step, t1 - step))
    res["kernels_us"] = {k: round(sum(v) / len(v), 2) for k, v in sorted(kernels.items(), key=lambda kv: -sum(kv[1]))}
    res["timeline_us"] = {k: [round(sum(a for a, _ in v) / len(v), 1), round(sum(b for _, b in v) / len(v), 1)]
                          for k, v in sorted(timeline.items(), key=lambda kv: sum(a for a, _ in kv[1]) / len(kv[1]))}
    res["kernel_launches_per_step"] = sum(len(v) for v in kernels.values()) / n

    # the all-pairs kernel alone: the benchmark's boxes after the step, config 3 (discs) and config 4 (IoU) shapes
    box = tds.ops.agent_boxes(runner.state, sim.get_agent_size())
    mask = torch.ones(B, A, dtype=torch.bool, device=dev)
    out = torch.empty(B, A, device=dev)
    rng = np.random.default_rng(0)

    def boxes(Bc, Ac, span):
        xy = rng.uniform(-span / 2, span / 2, (Bc, Ac, 2))
        return torch.tensor(np.concatenate([xy, np.tile([4.97, 2.04], (Bc, Ac, 1)), rng.uniform(0, 6.28, (Bc, Ac, 1))], -1),
                            dtype=torch.float32, device=dev)
    b3, b4 = boxes(512, 128, 300.0), boxes(64, 512, 120.0)
    o3, o4 = torch.empty(512, 128, device=dev), torch.empty(64, 512, device=dev)
    m3, m4 = torch.ones(512, 128, dtype=torch.bool, device=dev), torch.ones(64, 512, dtype=torch.bool, device=dev)
    res["allpairs_us"] = {
        "discs_1024x64_bench": graph_us(lambda: tds.ops.collision_allpairs(box, box, mask, out=out)),
        "discs_512x128_config3": graph_us(lambda: tds.ops.collision_allpairs(b3, b3, m3, out=o3)),
        "iou_64x512_config4": graph_us(lambda: tds.ops.collision_allpairs(b4, b4, m4, tds._lib.METRIC_IOU, out=o4)),
    }
    res["allpairs_us"] = {k: round(v, 2) for k, v in res["allpairs_us"].items()}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
