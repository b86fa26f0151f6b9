"""Host driver of the per-step hot path: the subset of the reference's `Simulator`
(torchdrivesim/simulator.py:280-1194) that the B200 kernels accelerate, with the same method names and
tensor conventions:

    step(action)            simulator.py:841-861   -> fused kinematic kernel
    render / render_egocentric  :920-1033          -> scene descriptor + raster kernel
    compute_collision       :1161-1194             -> ONE all-pairs launch instead of a Python loop over agents
    compute_offroad         :1035-1044             -> grid-accelerated point-to-mesh kernel

    npc_controller.advance_npcs :854 (+ :54-124, behavior/replay.py:46-107) -> one replay / spawn / despawn launch

    waypoint_goals.step     :860-861 (+ goals.py:159-217) -> one launch; observation noise: observation_noise.py

The lanelet-based wrong-way loss, the IAI / heuristic behaviour models and the map-from-log noise are out of scope (DESIGN.md §8).
"""
import copy as _copy
from dataclasses import dataclass, field
from enum import Enum
from typing import Dict, List, Optional, Tuple, Union

import math
import torch
from torch import Tensor

from . import _lib, ops
from .kinematic import KinematicModel
from .maps import MapSet, StaticMap
from .mesh import B200BirdviewMeshGenerator
from .goals import WaypointGoal
from .npc import NPCController
from .observation_noise import ObservationNoise
from .rendering import B200RendererConfig, BirdviewRenderer, RendererConfig, Resolution, renderer_from_config


class CollisionMetric(Enum):
    """Subset of simulator.py:27-34 that has a GPU kernel."""
    discs = 'discs'
    iou = 'iou'


@dataclass
class TorchDriveConfig:
    """Same fields as simulator.py:37-51 where they apply to the hot path."""
    renderer: RendererConfig = field(default_factory=B200RendererConfig)
    single_agent_rendering: bool = False
    collision_metric: CollisionMetric = CollisionMetric.discs
    offroad_threshold: float = 0.5
    waypoint_removal_threshold: float = 2.0    # how close an agent must get to a waypoint to achieve it
    left_handed_coordinates: bool = False


class Simulator:
    def __init__(self, road_mesh: Union[StaticMap, MapSet], kinematic_model: KinematicModel, agent_size: Tensor,
                 initial_present_mask: Tensor, cfg: TorchDriveConfig, renderer: Optional[BirdviewRenderer] = None,
                 birdview_mesh_generator: Optional[B200BirdviewMeshGenerator] = None, internal_time: int = 0,
                 traffic_controls: Optional[Dict[str, object]] = None, agent_types: Optional[Tensor] = None,
                 agent_type_names: Optional[List[str]] = None, npc_controller: Optional[NPCController] = None,
                 waypoint_goals: Optional[WaypointGoal] = None, observation_noise_model: Optional[ObservationNoise] = None):
        self.road_mesh = road_mesh if isinstance(road_mesh, MapSet) else MapSet([road_mesh])
        self.kinematic_model = kinematic_model
        self.agent_size = agent_size
        self.present_mask = initial_present_mask
        self._agent_types = agent_type_names or ['vehicle']
        self.agent_type = torch.zeros_like(initial_present_mask).long() if agent_types is None else agent_types
        self._batch_size = initial_present_mask.shape[0]
        self.cfg = cfg
        self.traffic_controls = traffic_controls
        self.internal_time = internal_time
        state = self.get_state()
        if npc_controller is None:
            # simulator.py:337-345: an empty controller, so that "all agents" are the controlled agents
            dev = initial_present_mask.device
            npc_controller = NPCController(npc_size=torch.zeros((self._batch_size, 0, 2), dtype=agent_size.dtype, device=dev),
                                           npc_state=torch.zeros((self._batch_size, 0, 4), dtype=state.dtype, device=dev),
                                           npc_present_mask=torch.zeros((self._batch_size, 0), dtype=torch.bool, device=dev),
                                           npc_types=torch.zeros((self._batch_size, 0), dtype=torch.long, device=dev),
                                           agent_type_names=self._agent_types)
        self.npc_controller = npc_controller
        self.waypoint_goals = waypoint_goals
        self.observation_noise_model = observation_noise_model or ObservationNoise()     # simulator.py:378-381
        if state.dim() != 3 or agent_size.shape[:2] != state.shape[:2] or initial_present_mask.shape != state.shape[:2]:
            raise _lib.TdsError("expected state [B,A,4], agent_size [B,A,2] and present mask [B,A]")
        if renderer is None:
            cfg.renderer.left_handed_coordinates = cfg.left_handed_coordinates
            renderer = renderer_from_config(cfg.renderer)
        self.renderer = renderer
        if cfg.left_handed_coordinates:
            self.kinematic_model.left_handed = True
        if birdview_mesh_generator is None:
            # note: like simulator.py:371, render_agent_direction from the config is NOT forwarded
            birdview_mesh_generator = B200BirdviewMeshGenerator(self.road_mesh, self.renderer.color_map,
                                                                self.renderer.rendering_levels,
                                                                batch_size=self._batch_size)
            birdview_mesh_generator.initialize_actors_mesh(self.get_all_agent_size(), self.get_all_agent_type(),
                                                           self.agent_types)
            if traffic_controls is not None:
                birdview_mesh_generator.initialize_traffic_controls_mesh(traffic_controls)
        self.birdview_mesh_generator = birdview_mesh_generator

    # ---- properties / getters (simulator.py:383-400, 561-640) ----------------------------------
    @property
    def agent_types(self) -> List[str]:
        return self._agent_types

    @property
    def action_size(self) -> int:
        return self.kinematic_model.action_size

    @property
    def batch_size(self) -> int:
        return self._batch_size

    @property
    def agent_count(self) -> int:
        return self.present_mask.shape[-1]

    def get_world_center(self) -> Tensor:
        return self.birdview_mesh_generator.world_center

    def get_state(self) -> Tensor:
        return self.kinematic_model.get_state()

    def get_agent_size(self) -> Tensor:
        return self.agent_size

    def get_agent_type(self) -> Tensor:
        return self.agent_type

    def get_present_mask(self) -> Tensor:
        return self.present_mask

    # ---- NPCs and "all agents" = controlled agents followed by NPCs (simulator.py:526-532, 681-728)
    @property
    def npc_count(self) -> int:
        return self.get_npc_size().shape[-2]

    def get_npc_state(self) -> Tensor:
        return self.npc_controller.get_npc_state()

    def get_npc_size(self) -> Tensor:
        return self.npc_controller.get_npc_size()

    def get_npc_present_mask(self) -> Tensor:
        return self.npc_controller.get_npc_present_mask()

    def get_npc_types(self) -> Tensor:
        return self.npc_controller.get_npc_types()

    def _with_npcs(self, agents: Tensor, npcs: Tensor, dim: int) -> Tensor:
        return agents if npcs.shape[1] == 0 else torch.cat([agents, npcs.to(agents.dtype)], dim=dim)

    def get_all_agent_state(self) -> Tensor:
        return self._with_npcs(self.get_state(), self.get_npc_state(), -2)

    def get_all_agent_size(self) -> Tensor:
        return self._with_npcs(self.get_agent_size(), self.get_npc_size(), -2)

    def get_all_agent_type(self) -> Tensor:
        return self._with_npcs(self.get_agent_type(), self.get_npc_types(), -1)

    def get_all_agent_present_mask(self) -> Tensor:
        return self._with_npcs(self.get_present_mask(), self.get_npc_present_mask(), -1)

    def get_traffic_controls(self):
        return self.traffic_controls

    # ---- waypoint goals (simulator.py:589-605)
    def get_waypoints(self, count: int = 1) -> Optional[Tensor]:
        return self.waypoint_goals.get_waypoints(count=count) if self.waypoint_goals is not None else None

    def get_waypoints_state(self) -> Optional[Tensor]:
        return self.waypoint_goals.state if self.waypoint_goals is not None else None

    def get_waypoints_mask(self, count: int = 1) -> Optional[Tensor]:
        return self.waypoint_goals.get_masks(count=count) if self.waypoint_goals is not None else None

    # ---- batch plumbing (simulator.py:401-517) -------------------------------------------------
    def to(self, device):
        self.kinematic_model = self.kinematic_model.to(device)
        self.agent_size = self.agent_size.to(device)
        self.agent_type = self.agent_type.to(device)
        self.present_mask = self.present_mask.to(device)
        if self.road_mesh.env_map is not None:
            self.road_mesh.env_map = self.road_mesh.env_map.to(device)
        self.birdview_mesh_generator = self.birdview_mesh_generator.to(device)
        if self.traffic_controls is not None:
            self.traffic_controls = {k: v.to(device) for k, v in self.traffic_controls.items()}
        self.npc_controller = self.npc_controller.to(device)
        self.waypoint_goals = self.waypoint_goals.to(device) if self.waypoint_goals is not None else None
        return self

    def copy(self):
        other = _copy.copy(self)
        other.kinematic_model = self.kinematic_model.copy()
        other.renderer = self.renderer.copy()
        other.birdview_mesh_generator = self.birdview_mesh_generator.copy()
        if self.traffic_controls is not None:
            other.traffic_controls = {k: v.copy() for k, v in self.traffic_controls.items()}
        other.npc_controller = self.npc_controller.copy()
        other.waypoint_goals = self.waypoint_goals.copy() if self.waypoint_goals is not None else None
        return other

    def extend(self, n: int, in_place: bool = True):
        """Multiplies the batch dimension by n: every environment is repeated n times in a row (simulator.py:443-478)."""
        if not in_place:
            return self.copy().extend(n, in_place=True)
        grow = lambda x: x.unsqueeze(1).expand((x.shape[0], n) + x.shape[1:]).reshape((n * x.shape[0],) + x.shape[1:])
        self.road_mesh = self.road_mesh.extend(n)
        self.agent_size, self.agent_type, self.present_mask = grow(self.agent_size), grow(self.agent_type), grow(self.present_mask)
        self.kinematic_model.extend(n)                      # kinematic models are modified in place
        self._batch_size *= n
        self.birdview_mesh_generator = self.birdview_mesh_generator.expand(n)
        if self.traffic_controls is not None:
            self.traffic_controls = {k: v.extend(n) for k, v in self.traffic_controls.items()}
        if self.waypoint_goals is not None:
            self.waypoint_goals = self.waypoint_goals.extend(n)
        self.npc_controller = self.npc_controller.extend(n)
        return self

    def select_batch_elements(self, idx: Tensor, in_place: bool = True):
        """Picks environments `idx` (the batch shard of one GPU in a multi-GPU run)."""
        other = self if in_place else self.copy()
        other.kinematic_model.select_batch_elements(idx)
        other.agent_size = other.agent_size[idx]
        other.agent_type = other.agent_type[idx]
        other.present_mask = other.present_mask[idx]
        other.road_mesh = other.road_mesh.select(idx)
        other.birdview_mesh_generator = other.birdview_mesh_generator.select_batch_elements(idx)
        if other.traffic_controls is not None:
            other.traffic_controls = {k: v.select_batch_elements(idx, in_place=in_place) for k, v in other.traffic_controls.items()}
        other.npc_controller = other.npc_controller.select_batch_elements(idx, in_place=in_place)
        if other.waypoint_goals is not None:
            other.waypoint_goals = other.waypoint_goals.select_batch_elements(idx, in_place=in_place)
        other._batch_size = int(idx.numel())
        return other

    # ---- hot path ---------------------------------------------------------------------------------
    def step(self, agent_action: Tensor) -> None:
        self.internal_time += 1
        if agent_action.dim() != 3 or agent_action.shape[0] != self.batch_size or agent_action.shape[-2] != self.agent_count:
            raise _lib.TdsError(f"action must be [B={self.batch_size}, A={self.agent_count}, Ac]")
        self.npc_controller.advance_npcs(self)             # simulator.py:854
        self.kinematic_model.step(agent_action)
        if self.traffic_controls is not None:
            for control in self.traffic_controls.values():
                control.step(self.internal_time)
        if self.waypoint_goals is not None:                # simulator.py:860-861
            self.waypoint_goals.step(self.get_state(), self.internal_time, threshold=self.cfg.waypoint_removal_threshold)

    def set_state(self, agent_state: Tensor, mask: Optional[Tensor] = None) -> None:
        if mask is None:
            self.kinematic_model.set_state(agent_state)
        else:
            self.kinematic_model.set_state(agent_state.where(mask.unsqueeze(-1), self.kinematic_model.get_state()))

    def update_present_mask(self, present_mask: Tensor) -> None:
        self.present_mask = present_mask

    def fit_action(self, future_state: Tensor, current_state: Optional[Tensor] = None) -> Tensor:
        return self.kinematic_model.fit_action(future_state=future_state, current_state=current_state)

    def _scene(self, camera_xy: Tensor, rendering_mask: Optional[Tensor], waypoints: Optional[Tensor],
               waypoints_rendering_mask: Optional[Tensor], custom_agent_colors: Optional[Tensor]):
        """The scene descriptor `render` hands to the renderer (simulator.py:961-990)."""
        n_cameras = camera_xy.shape[-2]
        present = self.get_all_agent_present_mask()
        if rendering_mask is not None:
            present = present.unsqueeze(-2).expand(-1, n_cameras, -1).logical_and(rendering_mask)
        else:
            present = present.unsqueeze(-2).expand(-1, n_cameras, -1)
        tl = self.traffic_controls.get('traffic_light') if self.traffic_controls is not None else None
        return self.birdview_mesh_generator.generate(
            n_cameras, agent_state=self.get_all_agent_state().detach()[:, None].expand(-1, n_cameras, -1, -1),
            present_mask=present, traffic_lights=tl, waypoints=waypoints,
            waypoints_rendering_mask=waypoints_rendering_mask, custom_agent_colors=custom_agent_colors)

    def render(self, camera_xy: Tensor, camera_psi: Tensor, res: Optional[Resolution] = None,
               rendering_mask: Optional[Tensor] = None, fov: Optional[float] = None, out: Optional[Tensor] = None,
               waypoints: Optional[Tensor] = None, waypoints_rendering_mask: Optional[Tensor] = None,
               custom_agent_colors: Optional[Tensor] = None, dtype=None, camera_sc: Optional[Tensor] = None) -> Tensor:
        """camera_xy BxNx2, camera_psi BxNx1 -> BxNx3xHxW (simulator.py:920-992); waypoints BxNxMx2 and their
        BxNxM mask draw goal-waypoint discs for the camera they belong to; custom_agent_colors BxNxAllx3 in [0,1]
        is the colour of each agent in each camera.  dtype: torch.float32 (default, the reference's image),
        torch.uint8 (the same values, 4x fewer bytes) or 'rank' (BxNxHxW draw ranks, see `renderer.rank_table`)."""
        if camera_sc is None:           # (sin, cos) of the camera orientation; the egocentric path hands it in
            camera_sc = torch.cat([torch.sin(camera_psi), torch.cos(camera_psi)], dim=-1)
        if camera_xy.dim() == 2:
            camera_xy, camera_sc = camera_xy.unsqueeze(1), camera_sc.unsqueeze(1)
        n_cameras = camera_xy.shape[-2]
        scene = self._scene(camera_xy, rendering_mask, waypoints, waypoints_rendering_mask, custom_agent_colors)
        img = self.renderer.render_frame(scene, camera_xy, camera_sc, res=res, fov=fov, out=out, dtype=dtype)
        return img.reshape((self.batch_size, n_cameras) + img.shape[1:])

    def _egocentric_cameras(self, ego_rotate: bool, visibility_matrix: Optional[Tensor], n_subsequent_waypoints: int):
        """Camera position, orientation and (sin, cos) of every controlled agent: one launch of ours instead of the
        slice + sin + cos + cat of simulator.py:1008-1017 (the heading is evaluated like every other heading of the path)."""
        state = self.get_state().detach()
        camera_psi = state[..., 2:3]
        camera_xy, camera_sc = ops.egocentric_cameras(state)
        if not ego_rotate:
            camera_psi = torch.ones_like(camera_psi) * (math.pi / 2)
            camera_sc = torch.cat([torch.sin(camera_psi), torch.cos(camera_psi)], dim=-1)
        rendering_mask = visibility_matrix
        if self.cfg.single_agent_rendering:
            rendering_mask = torch.eye(self.agent_count, dtype=torch.bool, device=state.device).unsqueeze(0).expand(
                self.batch_size, -1, -1)
        waypoints = waypoints_mask = None
        if self.waypoint_goals is not None:
            waypoints, waypoints_mask = self.waypoint_goals.get_waypoints_and_masks(count=n_subsequent_waypoints)
        return camera_xy, camera_psi, camera_sc, rendering_mask, waypoints, waypoints_mask

    def render_egocentric(self, ego_rotate: bool = True, res: Optional[Resolution] = None, fov: Optional[float] = None,
                          visibility_matrix: Optional[Tensor] = None, out: Optional[Tensor] = None,
                          n_subsequent_waypoints: int = 1, custom_agent_colors: Optional[Tensor] = None,
                          dtype=None) -> Tensor:
        """One camera per agent -> BxAx3xHxW (simulator.py:994-1033); with waypoint goals every agent sees the discs of
        its next `n_subsequent_waypoints` collections; custom_agent_colors BxAxAllx3: the colours agents see each
        other as."""
        camera_xy, camera_psi, camera_sc, rendering_mask, waypoints, waypoints_mask = self._egocentric_cameras(
            ego_rotate, visibility_matrix, n_subsequent_waypoints)
        return self.render(camera_xy, camera_psi, rendering_mask=rendering_mask, res=res, fov=fov, out=out,
                           waypoints=waypoints, waypoints_rendering_mask=waypoints_mask,
                           custom_agent_colors=custom_agent_colors, dtype=dtype, camera_sc=camera_sc)

    def render_egocentric_to_host(self, host_out: Tensor, chunk_envs: int = 128, res: Optional[Resolution] = None,
                                  fov: Optional[float] = None, ego_rotate: bool = True,
                                  visibility_matrix: Optional[Tensor] = None, n_subsequent_waypoints: int = 1,
                                  custom_agent_colors: Optional[Tensor] = None) -> Tensor:
        """`render_egocentric` delivered into a PINNED host tensor: [B,A,3,H,W] float32 (the reference's image),
        [B,A,3,H,W] uint8 (the same values as bytes: the pixels are integers in [0,255], rendering/cv2.py:50, so
        nothing is lost and a PCIe-bound consumer gets 4x the frames) or [B,A,H,W] uint8 with dtype 'rank' semantics
        when `host_out` has no channel dimension.  Environments are rendered in chunks into two device buffers while
        the previous chunk is copied out on a side stream, so the transfer overlaps the raster kernel.  Returns
        `host_out` (valid once the current stream is synchronised)."""
        res = self.renderer.res if res is None else res
        camera_xy, camera_psi, cam_sc, rendering_mask, waypoints, waypoints_mask = self._egocentric_cameras(
            ego_rotate, visibility_matrix, n_subsequent_waypoints)
        dev = camera_xy.device
        B, A = camera_xy.shape[0], camera_xy.shape[1]
        rank = host_out.dim() == 4
        tail = (res.height, res.width) if rank else (3, res.height, res.width)
        if tuple(host_out.shape) != (B, A) + tail or not host_out.is_pinned() or \
                host_out.dtype not in ((torch.uint8,) if rank else (torch.float32, torch.uint8)):
            raise _lib.TdsError("host_out must be a pinned tensor: float32 / uint8 [B,A,3,H,W] or uint8 [B,A,H,W] (draw ranks)")
        dtype = 'rank' if rank else host_out.dtype
        cam_xy = camera_xy.contiguous()
        scene = self._scene(cam_xy, rendering_mask, waypoints, waypoints_mask, custom_agent_colors)
        chunk = max(1, min(chunk_envs, B))
        key = ((chunk, A) + tail, host_out.dtype)
        if getattr(self, "_h2d_key", None) != key:
            self._h2d_bufs = [torch.empty(key[0], dtype=host_out.dtype, device=dev) for _ in range(2)]
            self._copy_stream = torch.cuda.Stream(device=dev)
            self._buf_free = [None, None]
            self._h2d_key = key
        main = torch.cuda.current_stream(dev)
        for i, b0 in enumerate(range(0, B, chunk)):
            b1 = min(b0 + chunk, B)
            buf = self._h2d_bufs[i % 2][: b1 - b0]
            if self._buf_free[i % 2] is not None:
                main.wait_event(self._buf_free[i % 2])          # the previous copy out of this buffer is done
            self.renderer.render_frame(scene.slice(b0, b1), cam_xy[b0:b1], cam_sc[b0:b1], res=res, fov=fov, out=buf, dtype=dtype)
            done = torch.cuda.Event()
            done.record(main)
            with torch.cuda.stream(self._copy_stream):
                self._copy_stream.wait_event(done)
                host_out[b0:b1].copy_(buf, non_blocking=True)
                free = torch.cuda.Event()
                free.record(self._copy_stream)
            self._buf_free[i % 2] = free
        main.wait_stream(self._copy_stream)
        return host_out

    # ---- non-visual observations (simulator.py:730-781) --------------------------------------------
    def get_all_agents_absolute(self) -> Tensor:
        """Bx(A+Npc)x6: x, y, psi, length, width, present (simulator.py:730-738)."""
        return torch.cat([self.get_all_agent_state()[..., :3], self.get_all_agent_size()[..., :2],
                          self.get_all_agent_present_mask().unsqueeze(-1).to(torch.float32)], dim=-1)

    def get_all_agents_relative(self, exclude_self: bool = True) -> Tensor:
        """BxAx(A+Npc-1 or A+Npc)x6: the pose of every agent and NPC in the frame of every controlled agent
        (simulator.py:748-781), one launch and no host synchronisation.  Differentiable, as in the reference: the
        gradient reaches the agent states (x, y, psi) and sizes (length, width) through get_all_agents_absolute."""
        return ops.agents_relative(self.get_all_agents_absolute(), self.agent_count, exclude_self)

    def get_nearest_agents_relative(self, k: int, max_distance: float = math.inf) -> Tuple[Tensor, Tensor]:
        """(BxAxkx6, BxAxk int64): the k nearest present agents and NPCs within `max_distance` of every controlled
        agent, sorted by distance (ties by index), in its frame as get_all_agents_relative(exclude_self=False) gives
        them, and their indices into get_all_agents_absolute; empty slots are zero with index -1 (see
        ops.nearest_agents_relative).  Differentiable like get_all_agents_relative."""
        return ops.nearest_agents_relative(self.get_all_agents_absolute(), k, self.agent_count, max_distance)

    def get_nearest_map_segments(self, k: int, max_distance: float = math.inf) -> Tuple[Tensor, Tensor, Tensor]:
        """(BxAxkx4, BxAxk int64, BxAxk int64): the k nearest lane-marking segments of the road mesh within
        `max_distance` of every controlled agent, sorted by distance to the segment (ties by index), as both endpoints in
        the agent's frame, with their palette classes and indices into `StaticMap.marking_segments`; empty slots are zero
        with class and index -1 (see ops.nearest_map_segments).  Differentiable: the gradient reaches the agent states
        (x, y, psi), and through the kinematic step the actions."""
        return ops.nearest_map_segments(self.get_state(), self.road_mesh, k, max_distance)

    def get_range_scan(self, n_rays: int, max_range: float = 50.0, markings: bool = True) -> Tuple[Tensor, Tensor, Tensor]:
        """(BxAxR, BxAxR int64, BxAxR int64): the distance along `n_rays` evenly spaced rays of every controlled agent (in
        its frame, ray 0 straight ahead) to the first box of another present agent or NPC, or with `markings` the first
        lane-marking segment of the road mesh, up to `max_range`; the kind of the hit (0 agent, 1 marking, -1 none) and
        its index into get_all_agents_absolute or `StaticMap.marking_segments` (see ops.range_scan).  Differentiable: the
        gradient reaches the states and sizes, and through the kinematic step the actions."""
        return ops.range_scan(self.get_all_agents_absolute(), n_rays, self.agent_count, max_range,
                              self.road_mesh if markings else None)

    def compute_time_to_collision(self, horizon: float = 5.0) -> Tuple[Tensor, Tensor]:
        """(BxA, BxA int64): the time to collision of every controlled agent within `horizon` seconds when every agent
        and NPC keeps its heading and speed, and the index of the agent or NPC it meets first (into
        get_all_agent_state), or (+inf, -1) (see ops.time_to_collision).  Differentiable: the gradient reaches the
        states and sizes of both agents of each contact, and through the kinematic step the actions."""
        return ops.time_to_collision(self.get_all_agent_state(), self.get_all_agent_size()[..., :2],
                                     self.get_all_agent_present_mask(), horizon, self.agent_count)

    # ---- noisy observations (simulator.py:663-679, 740-746, 784-821): what every agent perceives of all agents
    def get_noisy_state(self) -> Tensor:
        return self.observation_noise_model.get_noisy_state(self)

    def get_noisy_agent_size(self) -> Tensor:
        return self.observation_noise_model.get_noisy_agent_size(self)

    def get_noisy_present_mask(self) -> Tensor:
        return self.observation_noise_model.get_noisy_present_mask(self)

    def get_noisy_all_agents_absolute(self) -> Tensor:
        """BxAx(A+Npc)x6: x, y, psi, length, width, present as perceived by each agent."""
        return torch.cat([self.get_noisy_state()[..., :3], self.get_noisy_agent_size()[..., :2],
                          self.get_noisy_present_mask()[..., None].to(torch.float32)], dim=-1)

    def get_noisy_all_agents_relative(self, exclude_self: bool = True) -> Tensor:
        """BxAx(A+Npc-1 or A+Npc)x6: the perceived agents in the frame of the perceiving agent's own perceived pose.
        Differentiable in the perceived states and sizes; with the base ObservationNoise they are views of the true
        ones, so the gradient reaches the agent states and sizes (the standard sensing model detaches its noisy
        states)."""
        return ops.agents_relative(self.get_noisy_all_agents_absolute(), exclude_self=exclude_self)

    def get_noisy_nearest_agents_relative(self, k: int, max_distance: float = math.inf) -> Tuple[Tensor, Tensor]:
        """get_nearest_agents_relative over what each agent perceives (get_noisy_all_agents_absolute), in the frame of
        its own perceived pose: an agent that it does not perceive (perceived present flag 0, e.g. occluded under
        StandardSensingObservationNoise) is not listed."""
        return ops.nearest_agents_relative(self.get_noisy_all_agents_absolute(), k, max_distance=max_distance)

    def compute_offroad(self, out: Optional[Tensor] = None) -> Tensor:
        """simulator.py:1035-1044: offroad_infraction_loss(...) * present mask.  `out`: see ops.offroad."""
        return ops.offroad(self.get_state(), self.get_agent_size(), self.road_mesh, self.cfg.offroad_threshold,
                           self.get_present_mask(), out=out)

    def compute_traffic_lights_violations(self) -> Tensor:
        """simulator.py:1046-1062: which agents run a red light (TrafficLightControl.compute_violation) times the
        present mask: BxA in the dtype of the state, 1.0 = violation (`violation * present.to(state.dtype)` there)."""
        state = self.get_state()
        tl = self.traffic_controls.get('traffic_light') if self.traffic_controls is not None else None
        if tl is None:
            return torch.zeros(state.shape[0], state.shape[1], dtype=state.dtype, device=state.device)
        box = ops.agent_boxes(state.detach(), self.get_agent_size()[..., :2])
        return ops.traffic_light_violation(box, tl.corners, tl.state, tl.allowed_states.index('red'),
                                           tl.violation_rear_factor, present=self.get_present_mask()).to(state.dtype)

    def compute_collision(self, out: Optional[Tensor] = None) -> Tensor:
        """simulator.py:1161-1194 for the `discs` and `iou` metrics, all agents in one launch.  `out`: see
        ops.collision_allpairs."""
        state, size = self.get_state(), self.get_agent_size()[..., :2]
        if state.shape[-2] == 0:
            return torch.zeros_like(state[..., 0])
        box = ops.agent_boxes(state, size)
        metric = _lib.METRIC_IOU if self.cfg.collision_metric == CollisionMetric.iou else _lib.METRIC_DISCS
        all_box = box
        if self.npc_count > 0:
            all_box = ops.agent_boxes(self.get_all_agent_state(), self.get_all_agent_size()[..., :2])
        return ops.collision_allpairs(box, all_box, self.get_all_agent_present_mask(), metric, ego_is_prefix=True, out=out)
