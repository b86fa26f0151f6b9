"""The lean parts of the graphed step keep their bits: the all-pairs discs kernel (row discs staged in shared memory) sums
and picks its maximum in exactly the order it always has; the general raster kernel behind the LEAN draw pass leaves at
once when its redo list is empty and renders the cameras on it otherwise; the graphed step, with collisions and offroad
on a second branch, equals the eager calls."""
import numpy as np
import pytest
import torch

from tests import util

pytestmark = pytest.mark.gpu


def _allpairs_in_kernel_order(ego, all_box, mask):
    """The all-pairs discs result from the element-wise pair kernel, reduced in the order of the all-pairs kernel: lane l
    of the row's warp takes columns l, l + 32, ... in turn, then the warp combines the lanes by xor butterflies (sum; the
    largest overlap, the lower column on ties)."""
    import torchdrivesim_b200 as tds
    B, A, N = ego.shape[0], ego.shape[1], all_box.shape[1]
    p = ego[:, :, None, :].expand(B, A, N, 5).contiguous()
    q = all_box[:, None, :, :].expand(B, A, N, 5).contiguous()
    o = tds.ops.collision_pairwise(p, q, tds._lib.METRIC_DISCS) * mask[:, None, :].to(torch.float32)
    K = (N + 31) // 32
    pad = K * 32 - N
    osum = torch.nn.functional.pad(o, (0, pad), value=0.0).view(B, A, K, 32)
    omax = torch.nn.functional.pad(o, (0, pad), value=float("-inf")).view(B, A, K, 32)
    s = torch.zeros(B, A, 32, dtype=torch.float32, device=ego.device)
    best = torch.full((B, A, 32), float("-inf"), device=ego.device)
    besti = torch.zeros(B, A, 32, dtype=torch.int64, device=ego.device)
    lane = torch.arange(32, device=ego.device)
    for k in range(K):
        s = s + osum[:, :, k]
        take = omax[:, :, k] > best
        best = torch.where(take, omax[:, :, k], best)
        besti = torch.where(take, k * 32 + lane, besti)
    for sh in (16, 8, 4, 2, 1):
        other = lane ^ sh
        s = s + s[..., other]
        ob, oi = best[..., other], besti[..., other]
        take = (ob > best) | ((ob == best) & (oi < besti))
        best, besti = torch.where(take, ob, best), torch.where(take, oi, besti)
    out = s[..., 0] - best[..., 0] if N > 0 else torch.zeros(B, A, device=ego.device)
    return out, besti[..., 0].to(torch.int32)


def _boxes(rng, B, N, spread, special):
    xy = rng.normal(0, spread, (B, N, 2))
    lw = np.tile(np.array(util.VEH[:2]), (B, N, 1)) * rng.uniform(0.3, 1.2, (B, N, 1))
    psi = rng.uniform(-np.pi, 2 * np.pi, (B, N, 1))
    box = np.concatenate([xy, lw, psi], -1).astype(np.float32)
    if special:
        box[:, ::7, 2:4] = 0.0                  # zero-size boxes: r = 0, 0 / 0 in the overlap
        box[:, 3::11, 2] = box[:, 3::11, 3]     # squares: the tie of torch.maximum / minimum
        box[:, 5::13, 4] = np.nan               # nan_to_num of the box
    return box


@pytest.mark.parametrize("B,A,N", [(1024, 64, 64), (5, 1, 1), (5, 31, 31), (5, 33, 33), (3, 128, 128), (4, 20, 33),
                                   (2, 70, 90), (1, 64, 3938)])
def test_allpairs_discs_matches_the_reduction_order(B, A, N):
    import torchdrivesim_b200 as tds
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(B * 1000 + A * 10 + N)
    all_box = torch.tensor(_boxes(rng, B, N, 6.0, special=N > 1), device=dev)
    mask = torch.tensor(rng.uniform(size=(B, N)) > 0.15, device=dev)
    ego = all_box[:, :A].contiguous()
    out, arg = tds.ops._allpairs_fwd(ego, all_box, mask, tds._lib.METRIC_DISCS, True)
    ref, ref_arg = _allpairs_in_kernel_order(ego, all_box, mask)
    torch.cuda.synchronize()
    assert (ref > 0).any() or N == 1, "the scene has no overlaps: the test would not see the sums"
    assert torch.equal(out, ref), f"max |diff| {float((out - ref).abs().max())}"
    assert torch.equal(arg, ref_arg)


def _sim(B, A, seed, bench_scene=False):
    """A clustered scene (agents see each other), or with `bench_scene` the benchmark's: agents on random road vertices
    of the whole map, whose cameras never go on the redo list."""
    import bench
    import torchdrivesim_b200 as tds
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(seed)
    m = util.load_map_np("carla_Town01")
    if bench_scene:
        state, size, _, _ = bench.synth_inputs(B, A, seed, 1)
        present = np.ones((B, A), bool)
    else:
        state, size, _, present = util.random_scene(m, B, A, rng, absent_p=0.1)
    town = tds.StaticMap.from_npz(util.map_path("carla_Town01"))
    km = tds.KinematicBicycle(left_handed=True)
    km.set_params(lr=torch.full((B, A), util.VEH[2], device=dev))
    km.set_state(torch.tensor(state, device=dev))
    sim = tds.Simulator(town, km, torch.tensor(size, device=dev), torch.tensor(present, device=dev),
                        tds.TorchDriveConfig(left_handed_coordinates=True))
    acts = torch.tensor(rng.uniform(-1, 1, (3, B, A, 2)).astype(np.float32), device=dev)
    return sim, acts


def _redo_counters(sim):
    """(cameras on the redo list, cameras the general kernel behind the draw pass pulled from its work counter) of the
    last birdview call: the work counters follow the per-environment primitives in the raster workspace
    (tds_raster_workspace_bytes: per-environment primitives | 8 int32 counters | the redo list)."""
    import torchdrivesim_b200 as tds
    B, N = sim.batch_size, sim.agent_count
    at = tds._lib.load().tds_raster_workspace_bytes(B, N, 0, 0) - 32 - B * N * 4
    counters = sim.birdview_mesh_generator._workspace[at:at + 32].view(torch.int32).cpu()
    return int(counters[4]), int(counters[1])


@pytest.mark.parametrize("clip_cap", [None, "4"])
def test_graphed_step_and_the_redo_list(monkeypatch, clip_cap):
    """The benchmark's scene puts no camera on the redo list, and then the general kernel behind the draw pass leaves
    before it pulls a camera.  With room for only 4 border-crossing faces per camera (TDS_RASTER_CLIP_CAP) cameras of a
    clustered scene go on the list and the general kernel captured behind the draw pass renders them.  Either way the
    graphed step equals the eager one without the hook."""
    import torchdrivesim_b200 as tds
    hook = clip_cap is not None
    eager, acts = _sim(64, 16, 11, bench_scene=not hook)
    graphed, _ = _sim(64, 16, 11, bench_scene=not hook)
    if hook:
        monkeypatch.setenv("TDS_RASTER_CLIP_CAP", clip_cap)
    runner = tds.GraphedHotPath(graphed)         # the hook is read when the launches are captured
    monkeypatch.delenv("TDS_RASTER_CLIP_CAP", raising=False)
    for t in range(acts.shape[0]):
        eager.step(acts[t])
        img_e, coll_e, off_e = eager.render_egocentric(), eager.compute_collision(), eager.compute_offroad()
        img_g, coll_g, off_g = runner.run(acts[t])
        torch.cuda.synchronize()
        listed, pulled = _redo_counters(graphed)
        listed_e, pulled_e = _redo_counters(eager)
        if hook:
            assert listed > listed_e, f"{listed} cameras on the redo list with the hook, {listed_e} without"
        else:
            assert listed == listed_e == 0, f"{listed} / {listed_e} cameras on the redo list"
        # an empty list: no camera pulled; else every listed camera and one last pull per warp that ran
        for n_listed, n_pulled in ((listed, pulled), (listed_e, pulled_e)):
            assert n_pulled == 0 if n_listed == 0 else n_pulled >= n_listed, (n_listed, n_pulled)
        assert torch.equal(runner.state, eager.get_state())
        assert torch.equal(img_g, img_e), f"image differs at step {t}"
        assert torch.equal(coll_g, coll_e) and torch.equal(off_g, off_e)
