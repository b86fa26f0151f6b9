"""Offroad corner triage: the per-map distance bound settles on-road corners without a search.  With the triage on
(default) and off (TDS_OFFROAD_TRIAGE=0) the forward gives bit-identical values and the backward bit-identical
gradients; the stored bound holds against the brute-force oracle."""
import ctypes

import numpy as np
import pytest
import torch

from tests import util

pytestmark = pytest.mark.gpu


def _bench_like(m, B, A, rng, displace=0.0):
    """bench.synth_inputs: agents on road vertices, uniform headings, vehicle boxes; then displaced by N(0, displace)."""
    xy = util.road_points(m, B * A, rng).reshape(B, A, 2)
    xy = xy + displace * rng.standard_normal((B, A, 2))
    state = np.concatenate([xy, rng.uniform(0, 2 * np.pi, (B, A, 1)), rng.uniform(0, 5, (B, A, 1))], -1).astype(np.float32)
    size = np.tile(np.array(util.VEH[:2], np.float32), (B, A, 1))
    return state, size


def _fwd(mapset, state, size, present, thr):
    """out [B,A] and face [B,A,4] straight from tds_offroad_fwd."""
    import torchdrivesim_b200 as tds
    lib = tds._lib.load()
    B, A = state.shape[:2]
    out = torch.empty(B, A, dtype=torch.float32, device=state.device)
    face = torch.empty(B, A, 4, dtype=torch.int32, device=state.device)
    handles, n_maps = mapset.handles(state.device)
    tds._lib.check(lib.tds_offroad_fwd(handles, n_maps, tds._lib.ptr(mapset.env_map_on(state.device)), tds._lib.ptr(state),
                                       tds._lib.ptr(size), tds._lib.ptr(present), B, A, float(thr), tds._lib.ptr(out),
                                       tds._lib.ptr(face), tds._lib.stream_ptr(state.device)))
    torch.cuda.synchronize()
    return out, face


def _both(monkeypatch, mapset, state, size, present, thr):
    monkeypatch.delenv("TDS_OFFROAD_TRIAGE", raising=False)
    on = _fwd(mapset, state, size, present, thr)
    monkeypatch.setenv("TDS_OFFROAD_TRIAGE", "0")
    off = _fwd(mapset, state, size, present, thr)
    monkeypatch.delenv("TDS_OFFROAD_TRIAGE")
    return on, off


def _assert_same(on, off):
    (out_on, face_on), (out_off, face_off) = on, off
    assert torch.equal(out_on.view(torch.int32), out_off.view(torch.int32))      # bit for bit
    settled = face_on < 0
    # searched corners keep the face of the search; a settled corner had a search result, and the search stops early
    # only at a face within the threshold
    assert torch.equal(face_on[~settled], face_off[~settled])
    return float(settled.float().mean())


@pytest.mark.parametrize("displace", [0.0, 3.0, 10.0])
@pytest.mark.parametrize("thr", [0.0, 0.5, 2.0])
def test_triage_is_bit_identical_bench_shape(monkeypatch, displace, thr):
    import torchdrivesim_b200 as tds
    rng = np.random.default_rng(int(10 * displace + 100 * thr))
    m = util.load_map_np("carla_Town01")
    B, A = 1024, 64
    state, size = _bench_like(m, B, A, rng, displace)
    state[0, :3, 0] = np.nan                      # NaN positions
    state[1, :3, 2] = np.nan                      # NaN headings
    state[2, :4, :2] = np.array([[-500, -500], [1e4, 0], [0, 3e4], [200, -40]], np.float32)   # off the grid
    present = rng.uniform(size=(B, A)) >= 0.1
    town = tds.StaticMap.from_npz(util.map_path("carla_Town01"))
    dev = torch.device("cuda")
    st, sz, pr = torch.tensor(state, device=dev), torch.tensor(size, device=dev), torch.tensor(present, device=dev)
    on, off = _both(monkeypatch, tds.MapSet([town]), st, sz, pr, thr)
    frac = _assert_same(on, off)
    if thr == 0.0:
        assert torch.equal(on[1], off[1])                 # nothing is settled at thr = 0
    if thr == 0.5 and displace == 0.0:
        assert frac > 0.6                                 # the benchmark's case: most corners need no search
    assert int(on[1][~pr].max()) == -1 and float(on[0][~pr].abs().max()) == 0.0


def test_triage_two_maps(monkeypatch):
    import torchdrivesim_b200 as tds
    rng = np.random.default_rng(5)
    names = ["carla_Town01", "carla_Town02"]
    B, A = 64, 32
    env_map = np.arange(B) % 2
    state = np.empty((B, A, 4), np.float32)
    size = np.empty((B, A, 2), np.float32)
    for i, name in enumerate(names):
        s, z = _bench_like(util.load_map_np(name), B, A, rng, 1.0)
        state[env_map == i], size[env_map == i] = s[env_map == i], z[env_map == i]
    maps = [tds.StaticMap.from_npz(util.map_path(n)) for n in names]
    dev = torch.device("cuda")
    mapset = tds.MapSet(maps, torch.tensor(env_map, dtype=torch.int32, device=dev))
    st, sz = torch.tensor(state, device=dev), torch.tensor(size, device=dev)
    for thr in (0.0, 0.5, 2.0):
        on, off = _both(monkeypatch, mapset, st, sz, None, thr)
        frac = _assert_same(on, off)
        assert (frac > 0.3) == (thr > 0.0)


@pytest.mark.parametrize("displace", [0.0, 3.0])
def test_triage_backward_identical(monkeypatch, displace):
    import torchdrivesim_b200 as tds
    rng = np.random.default_rng(7)
    m = util.load_map_np("carla_Town01")
    state, size = _bench_like(m, 16, 64, rng, displace)
    present = torch.tensor(rng.uniform(size=(16, 64)) >= 0.1, device="cuda")
    town = tds.MapSet([tds.StaticMap.from_npz(util.map_path("carla_Town01"))])
    res = []
    for triage in ("1", "0"):
        monkeypatch.setenv("TDS_OFFROAD_TRIAGE", triage)
        st = torch.tensor(state, device="cuda").requires_grad_(True)
        sz = torch.tensor(size, device="cuda").requires_grad_(True)
        out = tds.ops.offroad(st, sz, town, 0.5, present)
        (out * torch.linspace(0.5, 2.0, out.numel(), device="cuda").view_as(out)).sum().backward()
        res.append((out.detach(), st.grad, sz.grad))
    for a, b in zip(*res):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    assert float(res[0][1].abs().max()) > 0


def test_triage_fused_rollout_identical(monkeypatch):
    """FusedRollout captures the offroad forward and backward in its graph: same loss and gradient either way (no
    collision term: its backward accumulates with float atomics)."""
    import torchdrivesim_b200 as tds
    rng = np.random.default_rng(3)
    m = util.load_map_np("carla_Town01")
    B, A, T = 4, 32, 4
    state, size = _bench_like(m, B, A, rng, 1.5)
    dev = torch.device("cuda")
    town = tds.StaticMap.from_npz(util.map_path("carla_Town01"))
    st, sz = torch.tensor(state, device=dev), torch.tensor(size, device=dev)
    pr = torch.ones(B, A, dtype=torch.bool, device=dev)
    lr = torch.full((B, A), util.VEH[2], device=dev)
    act = torch.tensor(rng.uniform(-1, 1, (T, B, A, 2)).astype(np.float32), device=dev)
    res = []
    for triage in ("1", "0"):
        monkeypatch.setenv("TDS_OFFROAD_TRIAGE", triage)
        ro = tds.FusedRollout(town, st, sz, lr, pr, T, offroad_threshold=0.5, left_handed=True, w_collision=0.0,
                              w_offroad=1.0, w_target=0.0)
        loss, grad = ro.run(act)
        res.append((float(loss), grad.clone()))
    assert res[0][0] == res[1][0] and res[0][0] > 0
    assert torch.equal(res[0][1], res[1][1])


def _bound_grid(town):
    import torchdrivesim_b200 as tds
    lib = tds._lib.load()
    h = town.handle(torch.device("cuda"))
    geom = np.zeros(4, np.float32)
    dims = np.zeros(2, np.int32)
    tds._lib.check(lib.tds_map_offroad_bound(h, geom.ctypes.data_as(ctypes.c_void_p), dims.ctypes.data_as(ctypes.c_void_p), None))
    codes = np.zeros((dims[1], dims[0]), np.uint8)
    tds._lib.check(lib.tds_map_offroad_bound(h, geom.ctypes.data_as(ctypes.c_void_p), dims.ctypes.data_as(ctypes.c_void_p),
                                             codes.ctypes.data_as(ctypes.c_void_p)))
    return geom, codes


@pytest.mark.parametrize("mapname", ["carla_Town01", "carla_Town10HD"])
def test_bound_holds_against_the_oracle(mapname):
    """Random points (and the corners) of sampled subcells: the oracle's fp32 distance is <= the stored bound."""
    from oracle import offroad as OF
    import torchdrivesim_b200 as tds
    m = util.load_map_np(mapname)
    town = tds.StaticMap.from_npz(util.map_path(mapname))
    (x0, y0, cs, unit), codes = _bound_grid(town)
    assert cs == 0.25 and unit == 1.0 / 64
    known = np.flatnonzero(codes.ravel() < 255)
    assert known.size > 0.05 * codes.size
    rng = np.random.default_rng(11)
    # subcells whose bound is small enough to settle a corner at the thresholds users set (<= 2.0 m^2) matter most
    small = np.flatnonzero(codes.ravel() <= 91)
    cells = np.concatenate([rng.choice(small, 1500, replace=False), rng.choice(known, 500, replace=False)])
    sy, sx = np.divmod(cells, codes.shape[1])
    uv = np.concatenate([rng.uniform(0, 1, (cells.size, 3, 2)), np.ones((cells.size, 1, 2))], 1)      # + the far corner
    px = (np.float32(x0) + ((sx[:, None] + uv[..., 0]) * cs).astype(np.float32)).astype(np.float32)
    py = (np.float32(y0) + ((sy[:, None] + uv[..., 1]) * cs).astype(np.float32)).astype(np.float32)
    d2, _ = OF.points_mesh_dist2(np.stack([px, py], -1).reshape(-1, 2), m["verts"], m["faces"])
    ub = codes.ravel()[cells].astype(np.float64) / 64.0
    assert (d2.reshape(cells.size, 4).astype(np.float64) <= (ub * ub)[:, None]).all()
