"""Range-scan observations on the GPU (ops.range_scan, tds_range_scan and its backward).

The forward is compared bit for bit (dist bits, kind, idx) with an eager torch brute force of its definition over every
candidate: the box edges of every other present agent and, with a map, the lane markings whose midpoint lies within
max_range + half their length (+ 1 m) of the origin, which cannot change a hit.  Every eager op rounds on its own, as
the definition asks; the headings' sin / cos are those of ops.egocentric_cameras, the library's double-precision
sincos rounded to float32.  The backward is compared with float64 autograd of the definition for the winning segments,
under the rounding-derived tolerance of test_gpu_observation_grads.check."""
import math

import numpy as np
import pytest
import torch

import torchdrivesim_b200 as tds
from tests import util
from tests.test_gpu_observation_grads import check
from torchdrivesim_b200 import ops

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
TOWNS = ("carla_Town01", "carla_Town02", "carla_Town10HD")
MAPS = {}
EMPTY = (1 << 63) - 1
SX = (0.5, -0.5, -0.5, 0.5)      # corner k of box2corners_th: (+,+), (-,+), (-,-), (+,-)
SY = (0.5, 0.5, -0.5, -0.5)


def town(name):
    if name not in MAPS:
        MAPS[name] = tds.StaticMap.from_npz(util.map_path(name))
    return MAPS[name]


def _bits(t):
    return t.contiguous().view(torch.int32)


# ------------------------------------------------------------------------------------------------ the definition
def ray_units(R, dtype=torch.float32):
    """[R,2]: (cos, sin)(2 pi r / R), reduced exactly to the nearest quarter turn (as sincospi does), then rounded."""
    out = []
    for r in range(R):
        q = (8 * r + R) // (2 * R)                 # the nearest quarter turn of 4r/R
        f = (4 * r - q * R) / (2 * R)              # the rest in half turns, |f| <= 1/4
        c, s = math.cos(math.pi * f), math.sin(math.pi * f)
        c, s = ((c, s), (-s, c), (-c, -s), (s, -c))[q % 4]
        out.append((c, s))
    return torch.tensor(out, dtype=torch.float64).to(dtype).to(DEV)


def sincos(absolute):
    """(sin psi, cos psi) [...] of the library (double precision, rounded to float32)."""
    st = torch.cat([absolute[..., :3], torch.zeros_like(absolute[..., :1])], -1)
    sc = ops.egocentric_cameras(st.contiguous())[1]
    return sc[..., 0], sc[..., 1]


def box_edges(absolute):
    """[B,N,4,4]: edge k = (corner k, corner (k + 1) % 4) of every box, the corner arithmetic of the offroad kernel."""
    s, c = (v[..., None] for v in sincos(absolute))
    x, y, l, w = (absolute[..., i, None] for i in (0, 1, 3, 4))
    ux = torch.tensor(SX, device=DEV) * l
    uy = torch.tensor(SY, device=DEV) * w
    px = (ux * c + uy * (-s)) + x
    py = (ux * s + uy * c) + y
    nx, ny = px.roll(-1, -1), py.roll(-1, -1)
    return torch.stack([px, py, nx, ny], -1)


def scan_ref(absolute, R, A, max_range, mapset=None, chunk=2048):
    """(dist, kind, idx, code) [B,A,R] of the definition; absolute [B,N,6] on the GPU."""
    B, N = absolute.shape[:2]
    mr = float(np.float32(max_range))
    units = ray_units(R)
    s, c = sincos(absolute)
    edges = box_edges(absolute).reshape(B, 4 * N, 4)
    j_of = torch.arange(4 * N, device=DEV) // 4
    env_map = torch.zeros(B, dtype=torch.int64) if mapset is None or mapset.env_map is None else mapset.env_map.long().cpu()
    word = torch.full((B, A, R), EMPTY, dtype=torch.int64, device=DEV)
    for mi in range(1 if mapset is None else len(mapset.maps)):
        bs = torch.nonzero(env_map == mi).flatten().to(DEV)
        if bs.numel() == 0 or A == 0:
            continue
        seg = None
        if mapset is not None:
            seg = mapset.maps[mi].marking_segments(DEV)[0].reshape(-1, 4)
            mid = 0.5 * (seg[:, :2].double() + seg[:, 2:].double())
            reach = mr + 0.5 * (seg[:, 2:].double() - seg[:, :2].double()).norm(dim=-1) + 1.0
        rows = bs.repeat_interleave(A), torch.arange(A, device=DEV).repeat(bs.numel())
        for r0 in range(0, rows[0].numel(), chunk):
            b, i = rows[0][r0:r0 + chunk], rows[1][r0:r0 + chunk]
            n = b.numel()
            o = absolute[b, i]
            finite = torch.isfinite(o[:, :3]).all(-1)
            cand = edges[b]                                                     # [n,4N,4]
            code = torch.arange(4 * N, device=DEV).expand(n, -1)
            ok = (absolute[b][:, :, 5] != 0)[:, j_of] & (j_of[None] != i[:, None])
            if seg is not None and seg.shape[0] > 0:
                near = (mid[None] - o[:, None, :2].double()).norm(dim=-1) <= reach[None]
                kmax = max(int(near.sum(1).max()), 1)
                order = torch.sort(near.to(torch.uint8), dim=1, descending=True, stable=True).indices[:, :kmax]
                cand = torch.cat([cand, seg[order]], 1)
                code = torch.cat([code, 4 * N + order], 1)
                ok = torch.cat([ok, near.gather(1, order)], 1)
            ok = ok & finite[:, None]
            dx = (c[b, i, None] * units[None, :, 0] - s[b, i, None] * units[None, :, 1])[..., None]      # [n,R,1]
            dy = (s[b, i, None] * units[None, :, 0] + c[b, i, None] * units[None, :, 1])[..., None]
            ex, ey = (cand[..., 2] - cand[..., 0])[:, None], (cand[..., 3] - cand[..., 1])[:, None]   # [n,1,K]
            wx, wy = (cand[..., 0] - o[:, 0, None])[:, None], (cand[..., 1] - o[:, 1, None])[:, None]
            den = dx * ey - dy * ex
            t = (wx * ey - wy * ex) / den
            u = (wx * dy - wy * dx) / den
            hit = (den != 0) & (u >= 0) & (u <= 1) & (t >= 0) & (t <= mr) & ok[:, None]
            t = torch.where(t == 0, 0.0, t)
            wd = torch.where(hit, (_bits(t).long() << 32) | code[:, None], EMPTY)
            word[b, i] = wd.amin(-1)
    none = word == EMPTY
    code = word & 0xFFFFFFFF
    dist = torch.where(none, mr, (word >> 32).int().view(torch.float32))
    kind = torch.where(none, -1, (code >= 4 * N).long())
    idx = torch.where(none, -1, torch.where(code >= 4 * N, code - 4 * N, code // 4))
    return dist, kind, idx, torch.where(none, -1, code)


def scene(rng, B, N, names=None, spread=8.0):
    """absolute [B,N,6]: agents clustered around a road vertex of the environment's map (names[b], Town01 by default)
    with random headings and vehicle-like sizes; some absent, some of zero size, some with NaN / inf x, y or psi, one
    1e4 m off the map."""
    names = names or ["carla_Town01"] * B
    rows = []
    for b in range(B):
        m = util.load_map_np(names[b])
        xy = util.road_points(m, 1, rng) + spread * rng.standard_normal((N, 2))
        xy[::5] = util.road_points(m, len(xy[::5]), rng)                     # exactly on road vertices
        size = np.stack([rng.uniform(3.5, 6.0, N), rng.uniform(1.6, 2.6, N)], -1)
        size[rng.uniform(size=N) < 0.1] = 0.0
        present = rng.uniform(size=N) > 0.15
        rows.append(np.concatenate([xy, rng.uniform(-7, 7, (N, 1)), size, present[:, None]], -1))
    a = np.stack(rows).astype(np.float32)
    a[0, 1, 0] = np.nan
    a[-1, 2, 1] = np.inf
    a[0, 3, 2] = np.nan
    a[-1, 4, :2] += 1e4
    return torch.tensor(a, device=DEV)


def _assert_same(got, ref):
    dist, kind, idx = got
    assert dist.dtype == torch.float32 and kind.dtype == torch.int64 and idx.dtype == torch.int64
    assert torch.equal(idx, ref[2])
    assert torch.equal(kind, ref[1])
    assert torch.equal(_bits(dist), _bits(ref[0]))


# ------------------------------------------------------------------------------------------------ forward
@pytest.mark.parametrize("markings", [True, False], ids=["markings", "agents_only"])
@pytest.mark.parametrize("max_range", [5.0, 50.0])
@pytest.mark.parametrize("R", [1, 3, 64, 256])
def test_forward_is_the_definition(R, max_range, markings):
    rng = np.random.default_rng(R * 100 + int(max_range) + markings)
    names = [TOWNS[b % 3] for b in range(6)]
    absolute = scene(rng, 6, 24, names)
    ms = tds.MapSet([town(n) for n in TOWNS], torch.tensor([b % 3 for b in range(6)], dtype=torch.int32))
    got = ops.range_scan(absolute, R, 18, max_range, ms if markings else None)
    ref = scan_ref(absolute, R, 18, max_range, ms if markings else None)
    _assert_same(got, ref)
    assert (got[1] == 0).any() and (got[1] == -1).any()
    if markings:
        assert (got[1] == 1).any()
    assert (got[1][0, 1] == -1).all() and (got[1][0, 3] == -1).all() and (got[1][-1, 2] == -1).all()   # NaN origins


def marking_map(segments):
    """A map whose lane markings are `segments` [(x0, y0, x1, y1)], each drawn as the strip of line_segments_to_mesh:
    faces (a,b,c),(b,c,d),(c,d,e),(d,e,f) with (c, d) the segment; plus a road square far away."""
    verts, faces, cat = [], [], []
    for x0, y0, x1, y1 in segments:
        p0, p1 = np.array([x0, y0]), np.array([x1, y1])
        tng = (p1 - p0) / max(np.linalg.norm(p1 - p0), 1e-9)
        nrm = np.array([-tng[1], tng[0]])
        v = len(verts)
        verts += [p0 - 0.1 * tng + 0.07 * nrm, p0 + 0.07 * nrm, p0, p1, p1 - 0.07 * nrm, p1 + 0.1 * tng - 0.07 * nrm]
        faces += [[v, v + 1, v + 2], [v + 1, v + 2, v + 3], [v + 2, v + 3, v + 4], [v + 3, v + 4, v + 5]]
        cat += [0] * 6
    v = len(verts)
    verts += [[500, 500], [510, 500], [500, 510], [510, 510]]
    faces += [[v, v + 1, v + 2], [v + 2, v + 1, v + 3]]
    cat += [1] * 4
    return tds.StaticMap(np.array(verts, np.float32), np.array(faces, np.int32), ["left_lane", "road"], np.array(cat))


ADVERSARIAL_SEGMENTS = [(-10, -5, 0, -5), (0, -5, 10, -5), (29, 29, 31, 31), (10, 0, 10, 2)]


def adversarial_scene():
    """absolute [1,12,6] (x, y, psi, length, width, present) of hand-placed agents:
    0 at the origin: ray +x runs through corner (10, 0) of box 1, the shared endpoint of its edges 1 and 2 (edge 2 is
      collinear with the ray, den == 0); box 2 is a copy of box 1 (equal t: the smaller code wins), and marking 3
      coincides with edge 1 (equal t: the agent edge wins);
    3 has zero size;  5 sits inside box 4;  6 sits on marking 2 (t = 0; the diagonal rays are parallel to it);
    7 looks at the shared endpoint (0, -5) of markings 0 and 1;  8 lies on the line of markings 0 and 1 (collinear rays);
    9 is 1e4 m off the map;  10 sits on the end of marking 1 (t = -0 for the rays pointing down);  11 is absent."""
    a = [[0, 0, 0, 4, 2, 1], [12, 1, 0, 4, 2, 1], [12, 1, 0, 4, 2, 1], [0, 10, 0.3, 0, 0, 1], [-20, 0.5, 0, 4, 3, 1],
         [-20, 0, 1.0, 4, 2, 1], [30, 30, 0, 4, 2, 1], [0, -15, 0, 4, 2, 1], [-20, -5, 0, 4, 2, 1], [1e4, 1e4, 0.2, 4, 2, 1],
         [10, -5, 0, 4, 2, 1], [2, 2, 0, 4, 2, 0]]
    return torch.tensor([a], dtype=torch.float32, device=DEV)


def test_marking_map_segments_are_the_strips():
    seg, _ = marking_map(ADVERSARIAL_SEGMENTS).marking_segments(DEV)
    assert torch.equal(seg.reshape(-1, 4).cpu(), torch.tensor(ADVERSARIAL_SEGMENTS, dtype=torch.float32))


@pytest.mark.parametrize("R", [4, 8, 256])
@pytest.mark.parametrize("markings", [True, False], ids=["markings", "agents_only"])
def test_adversarial_cases(R, markings):
    absolute = adversarial_scene()
    ms = tds.MapSet([marking_map(ADVERSARIAL_SEGMENTS)]) if markings else None
    dist, kind, idx = ops.range_scan(absolute, R, None, 50.0, ms)
    _assert_same((dist, kind, idx), scan_ref(absolute, R, 12, 50.0, ms))
    # agent 0, ray +x: edge 1 of box 1 at t = 10 (box 2 ties, marking 3 ties: the smaller code wins)
    assert float(dist[0, 0, 0]) == 10.0 and int(kind[0, 0, 0]) == 0 and int(idx[0, 0, 0]) == 1
    assert not ((kind == 0) & (idx == 3)).any()             # zero size
    assert not ((kind == 0) & (idx == 11)).any()            # absent
    assert (kind[0, 9] == -1).all() and (dist[0, 9] == 50.0).all()
    assert (kind[0, 5] == 0).all() and (idx[0, 5] == 4).all()  # inside box 4: every ray hits it
    if markings:
        on = (kind[0, 6] == 1) & (idx[0, 6] == 2)
        assert on.sum() >= R - 2 and (dist[0, 6][on] == 0).all() and (_bits(dist) >= 0).all()   # no -0
        if R % 4 == 0:                                       # ray 1 of agent 7 points exactly at (0, -5)
            assert float(dist[0, 7, R // 4]) == 10.0 and int(kind[0, 7, R // 4]) == 1 and int(idx[0, 7, R // 4]) == 0
        down = kind[0, 10] == 1
        assert down.any() and (dist[0, 10][down] == 0).all()


@pytest.mark.parametrize("R", [1, 3, 64])
def test_origin_far_off_the_map_and_env_map(R):
    rng = np.random.default_rng(R)
    absolute = scene(rng, 3, 16, ["carla_Town02"] * 3)
    absolute[1, :, :2] += 3e3
    ms = tds.MapSet([town("carla_Town02"), town("carla_Town01")], torch.tensor([0, 1, 0], dtype=torch.int32))
    _assert_same(ops.range_scan(absolute, R, 12, 50.0, ms), scan_ref(absolute, R, 12, 50.0, ms))
    dist, kind, idx = ops.range_scan(torch.zeros(3, 0, 6, device=DEV), R, None, 5.0, ms)
    assert dist.shape == kind.shape == idx.shape == (3, 0, R)


def test_config2_scale_is_the_definition():
    """1024 environments x 64 agents on Town01 at road positions (bench.py's inputs), 64 rays, 50 m."""
    import bench
    state, size, _, _ = bench.synth_inputs(1024, 64, 0, 1)
    absolute = torch.tensor(np.concatenate([state[..., :3], size, np.ones_like(size[..., :1])], -1), device=DEV)
    ms = tds.MapSet([town("carla_Town01")])
    got = ops.range_scan(absolute, 64, None, 50.0, ms)
    ref = scan_ref(absolute, 64, 64, 50.0, ms, chunk=4096)
    _assert_same(got, ref)
    assert float((got[1] >= 0).float().mean()) > 0.5


# ------------------------------------------------------------------------------------------------ backward
def grad_ref(absolute, R, A, kind, code, g, mapset=None):
    """float64 autograd of the definition with the winners fixed -> (d absolute [B,N,6], S [B,N,6]: the sum of the
    absolute products entering each element, inflated by the conditioning of den, t and u)."""
    B, N = absolute.shape[:2]
    x = absolute.double().clone().requires_grad_()
    bb, ii, rr = torch.nonzero(kind >= 0, as_tuple=True)
    cd = code[bb, ii, rr]
    agent = kind[bb, ii, rr] == 0
    j, k = (cd // 4).clamp(max=N - 1), cd % 4
    o = x[bb, ii]
    un = ray_units(R, torch.float64)[rr]
    cs, sn = torch.cos(o[:, 2]), torch.sin(o[:, 2])
    dx, dy = cs * un[:, 0] - sn * un[:, 1], sn * un[:, 0] + cs * un[:, 1]
    a = x[bb, j]
    ca, sa = torch.cos(a[:, 2]), torch.sin(a[:, 2])
    sxt, syt = torch.tensor(SX, dtype=torch.float64, device=DEV), torch.tensor(SY, dtype=torch.float64, device=DEV)

    def corner(kk):
        ux, uy = sxt[kk] * a[:, 3], syt[kk] * a[:, 4]
        return ux * ca - uy * sa + a[:, 0], ux * sa + uy * ca + a[:, 1], ux, uy

    c0x, c0y, ux0, uy0 = corner(k)
    c1x, c1y, ux1, uy1 = corner((k + 1) % 4)
    if mapset is not None:
        env = torch.zeros(B, dtype=torch.int64, device=DEV) if mapset.env_map is None else mapset.env_map.long().to(DEV)
        seg = torch.zeros(bb.numel(), 4, dtype=torch.float64, device=DEV)
        for mi, m in enumerate(mapset.maps):
            sm = m.marking_segments(DEV)[0].reshape(-1, 4).double()
            sel = ~agent & (env[bb] == mi)
            seg[sel] = sm[(cd[sel] - 4 * N)]
        c0x, c0y = torch.where(agent, c0x, seg[:, 0]), torch.where(agent, c0y, seg[:, 1])
        c1x, c1y = torch.where(agent, c1x, seg[:, 2]), torch.where(agent, c1y, seg[:, 3])
    ex, ey, wx, wy = c1x - c0x, c1y - c0y, c0x - o[:, 0], c0y - o[:, 1]
    den = dx * ey - dy * ex
    t = (wx * ey - wy * ex) / den
    gg = g[bb, ii, rr].double()
    (t * gg).sum().backward()
    with torch.no_grad():
        ad = den.abs()
        Q = gg.abs() / ad * (1 + (dx * ey).abs() / ad + (dy * ex).abs() / ad)
        T = t.abs() + ((wx * ey).abs() + (wy * ex).abs()) / ad
        Uc = ((wx * dy).abs() + (wy * dx).abs()) / ad
        u = (wx * dy - wy * dx) / den
        S = torch.zeros(B, N, 6, dtype=torch.float64, device=DEV)
        S[:, :, :3].index_put_((bb, ii), torch.stack([ey.abs() * Q, ex.abs() * Q, T * ((dx * ex).abs() + (dy * ey).abs()) * Q], -1),
                               accumulate=True)
        for wt, ux, uy in (((1 - u).abs() + Uc, ux0, uy0), (u.abs() + Uc, ux1, uy1)):
            gx, gy = ey.abs() * Q * wt, ex.abs() * Q * wt
            terms = torch.stack([gx, gy, gx * ((ux * sa).abs() + (uy * ca).abs()) + gy * ((ux * ca).abs() + (uy * sa).abs()),
                                 0.5 * (gx * ca.abs() + gy * sa.abs()), 0.5 * (gx * sa.abs() + gy * ca.abs())], -1)
            terms = torch.where(agent[:, None], terms, 0.0)
            S[:, :, :5].index_put_((bb, j), terms, accumulate=True)
    return x.grad, S


@pytest.mark.parametrize("R,max_range,markings", [(64, 50.0, True), (16, 5.0, True), (256, 50.0, False), (3, 50.0, True)])
def test_backward_vs_float64_autograd(R, max_range, markings):
    rng = np.random.default_rng(200 + R)
    absolute = scene(rng, 4, 24)
    absolute = torch.where(torch.isfinite(absolute), absolute, 0.0)
    ms = tds.MapSet([town("carla_Town01")]) if markings else None
    x = absolute.clone().requires_grad_()
    dist, kind, idx = ops.range_scan(x, R, 20, max_range, ms)
    _, ref_kind, _, code = scan_ref(absolute, R, 20, max_range, ms)
    assert torch.equal(kind, ref_kind) and (kind == 0).any()
    g = torch.tensor(rng.standard_normal((4, 20, R)).astype(np.float32), device=DEV)
    got, = torch.autograd.grad(dist, x, g)
    assert (got[..., 5] == 0).all()
    ref, S = grad_ref(absolute, R, 20, kind, code, g, ms)
    check(got, ref, S, terms=20 * R + R)
    again = ops._range_scan_bwd(absolute, R, 20, ms, kind, idx, g)
    assert torch.equal(_bits(again), _bits(got))


def test_rays_without_a_hit_contribute_nothing():
    rng = np.random.default_rng(9)
    absolute = scene(rng, 2, 16)
    ms = tds.MapSet([town("carla_Town01")])
    x = absolute.clone().requires_grad_()
    dist, kind, idx = ops.range_scan(x, 64, 12, 5.0, ms)
    none = kind == -1
    assert none.any() and (~none).any()
    g = torch.randn(2, 12, 64, device=DEV)
    g[none] = math.nan
    got, = torch.autograd.grad(dist, x, g)
    finite_rows = torch.isfinite(absolute).all(-1)
    assert torch.isfinite(got[finite_rows]).all()
    g0 = torch.where(none, 0.0, g)
    assert torch.equal(_bits(got), _bits(ops._range_scan_bwd(absolute, 64, 12, ms, kind, idx, g0)))
    zero = ops._range_scan_bwd(absolute, 64, 12, ms, torch.full_like(kind, -1), idx, g)
    assert (zero == 0).all()


# ------------------------------------------------------------------------------------------------ Simulator, graphs
def test_simulator_range_scan_and_its_gradient_reach_the_actions():
    rng = np.random.default_rng(3)
    name = "carla_Town01"
    m = util.load_map_np(name)
    B, A = 2, 8
    state, size, _, present = util.random_scene(m, B, A, rng, spread=6.0)
    km = tds.KinematicBicycle(left_handed=True)
    km.set_params(lr=torch.full((B, A), util.VEH[2], device=DEV))
    km.set_state(torch.tensor(state, device=DEV))
    sim = tds.Simulator(town(name), km, torch.tensor(size, device=DEV), torch.tensor(present, device=DEV),
                        tds.TorchDriveConfig(left_handed_coordinates=True))
    action = torch.tensor(rng.uniform(-1, 1, (B, A, 2)).astype(np.float32), device=DEV, requires_grad=True)
    sim.step(action)
    dist, kind, idx = sim.get_range_scan(32, 30.0)
    ref = ops.range_scan(sim.get_all_agents_absolute(), 32, sim.agent_count, 30.0, sim.road_mesh)
    for a, b in zip((dist, kind, idx), ref):
        assert torch.equal(a, b)
    assert (kind == 0).any() and (kind == 1).any()
    assert not (sim.get_range_scan(32, 30.0, markings=False)[1] == 1).any()
    dist.sum().backward()
    assert action.grad is not None and torch.isfinite(action.grad).all() and (action.grad != 0).any()


def test_cuda_graph_capture_replays_the_eager_result():
    rng = np.random.default_rng(4)
    absolute = scene(rng, 4, 24)
    ms = tds.MapSet([town("carla_Town01")])
    eager = ops._range_scan_fwd(absolute, 48, 20, 30.0, ms)
    g_in = torch.randn(4, 20, 48, device=DEV)
    eager_bwd = ops._range_scan_bwd(absolute, 48, 20, ms, eager[1], eager[2], g_in)
    static = absolute.clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ops._range_scan_fwd(static, 48, 20, 30.0, ms)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = ops._range_scan_fwd(static, 48, 20, 30.0, ms)
        gout = ops._range_scan_bwd(static, 48, 20, ms, out[1], out[2], g_in)
    static.copy_(torch.zeros_like(absolute))
    graph.replay()
    static.copy_(absolute)
    graph.replay()
    torch.cuda.synchronize()
    for a, b in zip(out, eager):
        assert torch.equal(_bits(a) if a.dtype == torch.float32 else a, _bits(b) if b.dtype == torch.float32 else b)
    assert torch.equal(_bits(gout), _bits(eager_bwd))
