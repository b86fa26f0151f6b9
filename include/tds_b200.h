/*
 * tds_b200.h — C ABI of the B200-native TorchDriveSim hot path (libtds_b200.so).
 *
 * The reference (inverted-ai/torchdrivesim 0.2.3) is pure Python: it has no FFI.  Its
 * "plugin API" for this path is constructor injection into `Simulator`
 * (torchdrivesim/simulator.py:299-309) plus module-level functions.  Each entry point below
 * replaces one of those Python call sites; the Python host layer (torchdrivesim_b200/*.py)
 * binds them with ctypes and mirrors the reference's classes.  See INTEGRATION.md.
 *
 * Conventions
 *   - every pointer named d_* is DEVICE memory on the current CUDA device, contiguous, in the
 *     reference's layout and dtype (fp32 state/boxes/images, uint8 masks, int32 indices);
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); calls only
 *     enqueue work: no host synchronisation, CUDA-graph capturable (except tds_map_create);
 *   - return value 0 = OK, otherwise an error code; tds_last_error() describes the last failure
 *     on the calling thread.  Data values never raise: NaNs are scrubbed where the reference
 *     scrubs them (simulator.py:1095-1103, infractions.py:171).
 *   - ownership: the caller owns all buffers; the library retains only tds_map_t handles.
 */
#ifndef TDS_B200_H
#define TDS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TDS_OK 0
#define TDS_ERR_INVALID_ARGUMENT 1
#define TDS_ERR_CUDA 2
#define TDS_ERR_UNSUPPORTED 3

#define TDS_MAX_CLASSES 32
#define TDS_MAX_AGENT_TYPES 8
#define TDS_MAX_TL_STATES 8
#define TDS_MAX_MAPS 8

int tds_version(void);
const char* tds_last_error(void);

/* ------------------------------------------------------------------------------------------
 * Kinematic state transition.  Replaces KinematicBicycle.step (kinematic.py:462-477),
 * BicycleNoReversing.step (kinematic.py:509-523) and the boolean-mask dispatch of
 * CompoundKinematicModel.step (kinematic.py:197-201); adds the unicycle the README names.
 * ---------------------------------------------------------------------------------------- */
#define TDS_MODEL_BICYCLE 0
#define TDS_MODEL_BICYCLE_NO_REVERSING 1
#define TDS_MODEL_UNICYCLE 2
#define TDS_MODEL_SIMPLE 3   /* SimpleKinematicModel.step, kinematic.py:362-367 (action = d state / dt, 4 values) */
#define TDS_MODEL_ORIENTED 4 /* OrientedKinematicModel.step, kinematic.py:384-389 (action xy in the agent frame)  */

typedef struct {
    float dt;               /* seconds */
    float max_acceleration; /* action[0] scale (kinematic.py:415) */
    float max_steering;     /* action[1] scale for the bicycle, float32(pi/2) by default */
    float max_yaw_rate;     /* action[1] scale for the unicycle */
    int32_t left_handed;    /* negate steering / yaw rate (kinematic.py:466-467) */
    float max_dx;           /* SIMPLE / ORIENTED action scales (kinematic.py:338-345): x, y */
    float max_dpsi;         /*   orientation */
    float max_dv;           /*   speed */
} tds_kinematic_params_t;

/* d_state [n,4] (x,y,psi,v), d_action [n,action_dim] with action_dim 2 or 4 (models 0-2 read the first two
 * values, models 3-4 need 4), d_lr [n], d_model [n] int32 or NULL (then uniform_model applies to every
 * agent), d_out_state [n,4] (may alias d_state). */
int tds_kinematic_step_fwd(const float* d_state, const float* d_action, int32_t action_dim, const float* d_lr,
                           const int32_t* d_model, int32_t uniform_model, int64_t n,
                           const tds_kinematic_params_t* params, float* d_out_state, void* stream);

/* Backward of the above.  d_grad_out [n,4]; outputs d_grad_state [n,4], d_grad_action [n,action_dim],
 * d_grad_lr [n] (any may be NULL). */
int tds_kinematic_step_bwd(const float* d_state, const float* d_action, int32_t action_dim, const float* d_lr,
                           const int32_t* d_model, int32_t uniform_model, int64_t n,
                           const tds_kinematic_params_t* params, const float* d_grad_out,
                           float* d_grad_state, float* d_grad_action, float* d_grad_lr, void* stream);

/* ------------------------------------------------------------------------------------------
 * Collisions.  Boxes are (x, y, length, width, psi).
 * ---------------------------------------------------------------------------------------- */
#define TDS_METRIC_DISCS 0 /* infractions.py:503-545 collision_detection_with_discs, 5 discs */
#define TDS_METRIC_IOU 1   /* infractions.py:307-324 iou_differentiable (fast)              */

/* Element-wise API of the reference functions: d_box1, d_box2 [p,5] -> d_out [p]. */
int tds_collision_pairwise_fwd(const float* d_box1, const float* d_box2, int64_t p, int32_t metric,
                               float* d_out, void* stream);
/* d_grad_out [p] -> d_grad_box1, d_grad_box2 [p,5] (either may be NULL).  The IoU gradient is the exact
 * gradient of intersection / union (boundary-integral form), which is what the reference's autograd
 * through its vertex formula evaluates. */
int tds_collision_pairwise_bwd(const float* d_box1, const float* d_box2, int64_t p, int32_t metric,
                               const float* d_grad_out, float* d_grad_box1, float* d_grad_box2, void* stream);

/* Fused Simulator.compute_collision (simulator.py:1161-1194, 1064-1109):
 *   out[b,i] = sum_j o(ego_i, all_j) m[b,j] - max_j o(ego_i, all_j) m[b,j]
 * d_ego_box [B,A,5], d_all_box [B,N,5], d_mask [B,N] uint8 (column presence),
 * d_out [B,A], d_argmax [B,A] int32 or NULL (index of the subtracted maximum, kept for bwd).
 * ego_is_prefix != 0 declares that ego agent i IS column i (the Simulator's layout); the IoU
 * metric then defines o(i,i) = 1 exactly (the reference's fp32 self-IoU is numerically chaotic). */
int tds_collision_allpairs_fwd(const float* d_ego_box, const float* d_all_box, const uint8_t* d_mask,
                               int32_t B, int32_t A, int32_t N, int32_t metric, int32_t ego_is_prefix,
                               float* d_out, int32_t* d_argmax, void* stream);
/* Backward of the above (both metrics).  d_grad_ego [B,A,5] is overwritten, d_grad_all [B,N,5] is
 * ACCUMULATED into (the caller zero-fills it). */
int tds_collision_allpairs_bwd(const float* d_ego_box, const float* d_all_box, const uint8_t* d_mask,
                               int32_t B, int32_t A, int32_t N, int32_t metric, int32_t ego_is_prefix,
                               const float* d_grad_out, const int32_t* d_argmax, float* d_grad_ego,
                               float* d_grad_all, void* stream);

/* ------------------------------------------------------------------------------------------
 * Traffic-light violations.  Replaces TrafficLightControl.compute_violation (traffic_controls.py:152-178)
 * with box2corners_with_rear_factor (_iou_utils.py:302-341) and the mask of
 * Simulator.compute_traffic_lights_violations (simulator.py:1046-1062):
 *   out[b,a] = present[b,a] and any over lights l of ( state[b,l] == red_state and
 *              area( rear `rear_factor` part of box[b,a]  intersected with  stop line l ) > 0 ).
 *   d_agent_box [B,A,5] (x, y, length, width, psi); d_tl_corners [B,L,4,2] in the corner order of
 *   box2corners_th (masked controls have all corners equal); d_tl_state [B,L] int32; d_present [B,A] uint8 or NULL;
 *   d_out [B,A] uint8.
 * ---------------------------------------------------------------------------------------- */
int tds_traffic_light_violation(const float* d_agent_box, const float* d_tl_corners, const int32_t* d_tl_state,
                                const uint8_t* d_present, int32_t B, int32_t A, int32_t L, int32_t red_state,
                                float rear_factor, uint8_t* d_out, void* stream);

/* ------------------------------------------------------------------------------------------
 * Replayed NPCs with spawning / despawning.  Replaces ReplayController.advance_npcs (behavior/replay.py:54-60)
 * + SpawnController.spawn_despawn_npcs (simulator.py:71-85) + utils.is_inside_polygon (utils.py:99-122):
 *   state, present <- replay[:, :, t_replay]                     (d_replay_states [B,Np,T,4], d_replay_present
 *                                                                 [B,Np,T] uint8 or NULL = all present; both NULL: keep)
 *   present &= inside the convex polygon d_exit_boundary [B,V,2]  (NULL: no despawning)
 *   spawn = d_spawn_masks[:, :, t_spawn] & !present; present |= spawn; state <- d_spawn_states[:, :, t_spawn] where spawn
 *                                                                (d_spawn_states [B,Np,Ts,4], d_spawn_masks [B,Np,Ts]; NULL: none)
 * d_npc_state [B,Np,4] and d_npc_present [B,Np] uint8 are updated in place.
 * ---------------------------------------------------------------------------------------- */
int tds_npc_advance(const float* d_replay_states, const uint8_t* d_replay_present, int32_t T, int32_t t_replay,
                    const float* d_exit_boundary, int32_t V, const float* d_spawn_states, const uint8_t* d_spawn_masks,
                    int32_t Ts, int32_t t_spawn, float* d_npc_state, uint8_t* d_npc_present, int32_t B, int32_t Np,
                    void* stream);

/* ------------------------------------------------------------------------------------------
 * Waypoint goals.  Replaces WaypointGoal.step (goals.py:159-217) and get_waypoints / get_masks (goals.py:33-105).
 *   d_waypoints [n_agents,N,M,2]: N collections of M waypoints per agent; d_mask [n_agents,N,M] uint8 (0 = padding or
 *   achieved); d_state [n_agents] int64 = current collection of each agent; d_agent_state [n_agents,4] (x, y, psi, v).
 * step:   if the agent is within `threshold` of a masked-in waypoint of its current collection, the collection's mask
 *         is cleared and the state advances (clamped to N-1); mask and state are updated in place.
 * gather: the next `count` collections of every agent -> d_out_waypoints [n_agents,count*M,2], d_out_mask
 *         [n_agents,count*M]; collections past the last one are zeros / masked out.
 * ---------------------------------------------------------------------------------------- */
int tds_waypoint_step(const float* d_agent_state, const float* d_waypoints, uint8_t* d_mask, int64_t* d_state,
                      int64_t n_agents, int32_t N, int32_t M, float threshold, void* stream);
int tds_waypoint_gather(const float* d_waypoints, const uint8_t* d_mask, const int64_t* d_state, int64_t n_agents,
                        int32_t N, int32_t M, int32_t count, float* d_out_waypoints, uint8_t* d_out_mask, void* stream);

/* ------------------------------------------------------------------------------------------
 * Aggregate infraction metrics of a step: the vector a multi-GPU job all-reduces (no reference counterpart: the
 * reference leaves the aggregation of compute_collision / compute_offroad to its callers).
 *   d_acc[0..5] (float64, accumulated in place) += sum of d_collision over present agents, sum of d_offroad,
 *   agents with collision > 0, agents with offroad > 0, present agents, agent slots n.  d_present [n] uint8 or NULL.
 * One launch, fixed reduction order (reproducible sums).
 * ---------------------------------------------------------------------------------------- */
int tds_infraction_metrics(const float* d_collision, const float* d_offroad, const uint8_t* d_present, int64_t n,
                           double* d_acc, void* stream);

/* ------------------------------------------------------------------------------------------
 * Glue of the per-step path and of differentiable rollouts: what the reference does with eager torch ops between its
 * hot functions, as single launches.
 * tds_agent_boxes:  d_state [n,4] (x, y, psi, v), d_size [n,2] (length, width) -> d_box [n,5] (x, y, length, width, psi),
 *                   the box layout of compute_collision (simulator.py:1161-1170); d_cam_sc [n,2] = (sin psi, cos psi) and
 *                   d_xy [n,2] = (x, y), the egocentric cameras of render_egocentric (simulator.py:961, 1017).  Any output
 *                   may be NULL.
 * tds_rollout_loss: d_acc[0..2] (float64, accumulated) += sum of d_collision [n], sum of d_offroad [n],
 *                   sum over agents of |xy - target|^2 (d_state [n,4], d_target_xy [n,2]); any input may be NULL.
 *                   One launch, fixed reduction order.
 * tds_rollout_grad: d loss / d state of one step of a rollout whose loss is  w_c sum collision + w_o sum offroad +
 *                   (w_t / 2) sum |xy - target|^2 :   d_grad_state [n,4] = d_grad_next (gradient arriving from the next
 *                   kinematic step, NULL: 0) + w_o d_grad_offroad (tds_offroad_bwd, [n,4]) + w_c (d_grad_box_ego +
 *                   d_grad_box_all)[x, y, psi] (tds_collision_allpairs_bwd, [n,5] each) + w_t (xy - target).
 * ---------------------------------------------------------------------------------------- */
int tds_agent_boxes(const float* d_state, const float* d_size, int64_t n, float* d_box, float* d_cam_sc, float* d_xy,
                    void* stream);
int tds_rollout_loss(const float* d_collision, const float* d_offroad, const float* d_state, const float* d_target_xy,
                     int64_t n, double* d_acc, void* stream);
int tds_rollout_grad(const float* d_grad_next, const float* d_grad_offroad, const float* d_grad_box_ego,
                     const float* d_grad_box_all, const float* d_state, const float* d_target_xy, float w_offroad,
                     float w_collision, float w_target, int64_t n, float* d_grad_state, void* stream);

/* ------------------------------------------------------------------------------------------
 * Non-visual observations.  Replaces Simulator.get_all_agents_relative (simulator.py:748-781) with
 * utils.relative (utils.py:71-79): for every origin agent i < A and every agent j < N of the same environment
 *   out = ( R(-psi_i) (xy_j - xy_i),  normalize_angle(psi_j - psi_i),  length_j, width_j, present_j ).
 *   d_absolute [B,N,6] (x, y, psi, length, width, present) as get_all_agents_absolute returns it; the first A
 *   agents are the origins.  d_out [B,A,N,6], or [B,A,N-1,6] with exclude_self (entry j == i removed; no
 *   boolean-mask indexing and hence no host synchronisation, unlike the reference).
 * ---------------------------------------------------------------------------------------- */
int tds_agents_relative(const float* d_absolute, int32_t B, int32_t A, int32_t N, int32_t exclude_self,
                        int32_t per_origin, float* d_out, void* stream);
/* per_origin != 0: d_absolute is [B,A,N,6], what each origin agent perceives (get_noisy_all_agents_relative,
 * simulator.py:784-821); the origin of row i is its own entry d_absolute[b,i,i]. */
int tds_agents_relative_bwd(const float* d_absolute, const float* d_grad_out, int32_t B, int32_t A, int32_t N,
                            int32_t exclude_self, int32_t per_origin, float* d_grad_absolute, void* stream);
/* The gradient of tds_agents_relative (autograd through utils.relative, utils.py:31-79): d_grad_out is the upstream
 * gradient in the layout of d_out, d_grad_absolute receives the gradient in the layout of d_absolute (every element is
 * written).  Per pair with (s, c) = sin / cos(-psi_i) and upstream row g: the observed agent j gets (c g0 + s g1,
 * -s g0 + c g1, g2, g3, g4, g5), the origin i gets (-(c g0 + s g1), -(-s g0 + c g1), g0 ry - g1 rx - g2, 0, 0, 0),
 * (rx, ry) being the pair's relative position.  Shared mode: agent n sums its observed terms over column n of every
 * origin row, plus, for n < A, its origin terms over its own row.  per_origin: entry [b,i,j != i] gets the observed
 * terms of row i, the origin entry [b,i,i] the origin terms of row i (plus its observed terms without exclude_self).
 * No atomics: two calls give bit-identical gradients.  d_absolute is re-read; the forward output is not needed. */
int tds_nearest_agents_relative(const float* d_absolute, int32_t B, int32_t A, int32_t N, int32_t k, int32_t per_origin,
                                float r2, float* d_out, int64_t* d_idx, void* stream);
/* The k nearest agents of every origin, as rows of tds_agents_relative without exclude_self.  d_absolute as above
 * (per_origin selects the mode), 1 <= k <= 64, r2 >= 0 (+inf: no distance limit).  For origin i and agent j != i, with
 * d = xy_j - xy_i in float32 and key = d.x*d.x + d.y*d.y (each operation rounded on its own, no FMA), j is eligible iff
 * present_j != 0 and key <= r2; a NaN key is never eligible, the origin's own present flag is not read.  Eligible
 * agents are ordered by (key, j) ascending.  d_out [B,A,k,6]: slot s holds the bits of tds_agents_relative's entry
 * [b,i,j] (exclude_self = 0) of the s-th agent j; d_idx [B,A,k] receives j.  Slots past the eligible agents are zero
 * with index -1.  No host synchronisation, no allocation. */
int tds_nearest_agents_relative_bwd(const float* d_absolute, const int64_t* d_idx, const float* d_grad_out, int32_t B,
                                    int32_t A, int32_t N, int32_t k, int32_t per_origin, float* d_grad_absolute,
                                    void* stream);
/* The gradient of tds_nearest_agents_relative through its filled slots (the selection is piecewise constant): d_idx
 * as the forward wrote it, d_grad_out [B,A,k,6], d_grad_absolute in the layout of d_absolute (every element is
 * written).  Each slot (i, s) with agent j contributes the per-pair terms of tds_agents_relative_bwd for the pair
 * (i, j): the observed terms to agent j, the origin terms to agent i (per_origin: to entries [b,i,j] and [b,i,i]).
 * A slot with index -1 (or any index that is not an agent other than i) is skipped, not multiplied by 0.  Shared mode
 * sums each agent's terms in an order fixed by the code, without atomics: two calls give bit-identical gradients. */

/* ------------------------------------------------------------------------------------------
 * Noisy observations.  Replaces StandardSensingObservationNoise (observation_noise.py:69-132):
 * sensing_noise:     d_out[b,a,e,:] = d_all_state[b,e,:] + d_eps[b,a,e,:] * deviation(|xy_a - xy_e|), deviation = 0.19 /
 *                    1.6 / 3.2 / 3.83 beyond 0.5 / 25 / 50 / 100 m (get_noisy_state; d_eps = standard normal deviates,
 *                    [B,A,N,4]; the first A of the N agents are the observers).
 * sensing_occlusion: d_out[b,a,e] = d_base_mask[b,e] and no third agent's circle (radius width/2) crosses the segment
 *                    from observer a to agent e (get_noisy_present_mask with utils.line_circle_intersection,
 *                    utils.py:139-187).  d_all_state [B,N,4], d_all_size [B,N,2], d_base_mask [B,N] uint8, d_out [B,A,N].
 * ---------------------------------------------------------------------------------------- */
int tds_sensing_noise(const float* d_all_state, const float* d_eps, int32_t B, int32_t A, int32_t N, float* d_out,
                      void* stream);
int tds_sensing_occlusion(const float* d_all_state, const float* d_all_size, const uint8_t* d_base_mask, int32_t B,
                          int32_t A, int32_t N, uint8_t* d_out, void* stream);

/* ------------------------------------------------------------------------------------------
 * Static map: triangle mesh + uniform grids, built once per map per GPU.  Replaces the
 * per-camera / per-corner expansion of the mesh (mesh.py:1147-1157, infractions.py:219-226).
 * ---------------------------------------------------------------------------------------- */
typedef struct tds_map tds_map_t;

/* Host inputs: verts [nv,2] f32, faces [nf,3] i32, face_class [nf] u8 (palette class of the face,
 * i.e. the category of its first vertex, cv2.py:58).  Cell sizes in metres (<= 0: defaults).
 * Synchronous (allocates and uploads).  Returns NULL on failure. */
tds_map_t* tds_map_create(const float* h_verts, int32_t nv, const int32_t* h_faces, int32_t nf,
                          const uint8_t* h_face_class, float raster_cell, float offroad_cell);
void tds_map_destroy(tds_map_t* map);

typedef struct {
    int32_t n_verts, n_faces;
    int32_t raster_gx, raster_gy, raster_records;
    int32_t offroad_gx, offroad_gy, offroad_entries;
    float raster_cell, offroad_cell;
    float min_x, min_y, max_x, max_y;
    int64_t device_bytes;
    int32_t raster_strips;   /* six-vertex strip records (four faces each), counted once per cell they are binned in */
    int32_t reserved;
} tds_map_info_t;
int tds_map_info(const tds_map_t* map, tds_map_info_t* out);
/* The offroad distance bound of a map (what tds_offroad_fwd uses to settle on-road corners without a search):
 * h_geom[4] = x0, y0 of the grid, subcell size, metres per code unit; h_dims[2] = gx, gy; h_codes [gy][gx] u8 or NULL.
 * Code q < 255: every point of the subcell lies within q * h_geom[3] metres of the mesh by the reference's fp32
 * distance; 255: unknown.  Synchronous copy. */
int tds_map_offroad_bound(const tds_map_t* map, float* h_geom, int32_t* h_dims, uint8_t* h_codes);

/* ------------------------------------------------------------------------------------------
 * Map observations: lane-marking segments.  The reference's line_segments_to_mesh (lanelet2.py:253-283) draws every
 * lane-marking segment [p0, p1] as four faces (a,b,c),(b,c,d),(c,d,e),(d,e,f) with c = p0 and d = p1.  Segment s of a
 * map is the s-th such strip in face order, as the greedy strip scan of tds_map_create finds it: four consecutive faces
 * of one class over six distinct finite vertices, listed in that order.  Its geometry is (c, d), its kind the strip's
 * palette class.  A map without such strips has no segment.
 * tds_map_segments: *h_count = S; h_seg [S][4] = (x0, y0, x1, y1) and h_kind [S] (either may be NULL).  Synchronous.
 * ---------------------------------------------------------------------------------------- */
int tds_map_segments(const tds_map_t* map, float* h_seg, uint8_t* h_kind, int32_t* h_count);
/* The k nearest segments of every agent, in its frame.  maps[d_env_map[b]] is the map of environment b (d_env_map NULL:
 * map 0), d_state [B,A,4] (x, y, psi, v), 1 <= k <= 256, r2 >= 0 (+inf: no distance limit).  For agent (x, y, psi) and
 * segment (x0, y0, x1, y1), in float32 with every operation rounded on its own (no FMA):
 *   e = p1 - p0, w = (x, y) - p0, l2 = ex*ex + ey*ey, t = l2 > 0 ? clamp((wx*ex + wy*ey) / l2, 0, 1) : 0 (IEEE division),
 *   q = w - t e, key = qx*qx + qy*qy.
 * A segment is eligible iff key <= r2 (a NaN key never is; an agent whose x or y is not finite has none).  Eligible
 * segments are ordered by (key, s).  Slot j: d_out [B,A,k,4] (16-byte aligned) = (rx0, ry0, rx1, ry1), both endpoints
 * in the agent's frame with the position arithmetic of tds_agents_relative: (s, c) = sincos(-psi), d = p - (x, y),
 * (c dx + (-s) dy, s dx + c dy); d_kind [B,A,k] the segment's class, d_idx [B,A,k] its s.  Leftover slots are zero with
 * kind and idx -1.  No host synchronisation, no allocation. */
int tds_nearest_map_segments(const tds_map_t* const* maps, int32_t n_maps, const int32_t* d_env_map, const float* d_state,
                             int32_t B, int32_t A, int32_t k, float r2, float* d_out, int64_t* d_kind, int64_t* d_idx,
                             void* stream);
/* The gradient of the above with respect to (x, y, psi) through the filled slots (the map is constant, the selection
 * piecewise constant): d_idx as the forward wrote it, d_grad_out [B,A,k,4], d_grad_state [B,A,4] (every element is
 * written; v gets 0).  Per endpoint with upstream (g0, g1): d x -= c g0 + s g1, d y -= -s g0 + c g1,
 * d psi += g0 ry - g1 rx.  A slot whose index is not a segment of the map is skipped, not multiplied by 0.  No atomics:
 * two calls give bit-identical gradients. */
int tds_nearest_map_segments_bwd(const tds_map_t* const* maps, int32_t n_maps, const int32_t* d_env_map,
                                 const float* d_state, const int64_t* d_idx, const float* d_grad_out, int32_t B, int32_t A,
                                 int32_t k, float* d_grad_state, void* stream);

/* ------------------------------------------------------------------------------------------
 * Range scan (no counterpart in the reference): the distance along R rays of every origin agent to the first agent box
 * edge or lane-marking segment.  d_absolute [B,N,6] (x, y, psi, length, width, present) as for tds_agents_relative; the
 * first A agents are the origins, whatever their present flag.  1 <= R <= 256, max_range finite and > 0.  maps /
 * n_maps / d_env_map as for tds_nearest_map_segments; n_maps = 0 (maps NULL): agents only.
 * Ray r of origin i: u = (float32 cospi(2r/R), float32 sinpi(2r/R)) (evaluated in double), (s, c) = sincos(psi_i),
 * d = (c ux - s uy, s ux + c uy), o = (x_i, y_i).  Candidates: edge k of every agent j != i with present_j != 0, from
 * corner k to corner (k + 1) % 4 in the corner order of box2corners_th (the corners of tds_offroad_fwd), code 4 j + k;
 * marking segment s of the map (tds_map_segments), code 4 N + s.  In float32, every operation rounded on its own:
 *   e = p1 - p0, w = p0 - o, den = dx*ey - dy*ex; den == 0: no hit; t = (wx*ey - wy*ex) / den, u = (wx*dy - wy*dx) / den
 *   (IEEE division); a hit iff 0 <= u <= 1 and 0 <= t <= max_range (a NaN never hits); a t of -0 counts as +0.
 * The winner is the smallest (bits(t) << 32 | code).  d_dist [B,A,R] = its t, or max_range without a hit; d_kind
 * [B,A,R] = 0 for an agent edge, 1 for a marking, -1 for none; d_idx [B,A,R] = j, s or -1.  An origin whose x, y or psi
 * is not finite hits nothing.  No host synchronisation, no allocation. */
int tds_range_scan(const tds_map_t* const* maps, int32_t n_maps, const int32_t* d_env_map, const float* d_absolute,
                   int32_t B, int32_t A, int32_t N, int32_t R, float max_range, float* d_dist, int64_t* d_kind,
                   int64_t* d_idx, void* stream);
/* The gradient of d_dist with respect to d_absolute (the map is constant, the selection piecewise constant): d_kind and
 * d_idx as the forward wrote them, d_grad_dist [B,A,R], d_grad_absolute [B,N,6] (every element is written; the present
 * column gets 0).  A ray reaches its origin's x, y, psi and, for an agent hit, the hit agent's x, y, psi, length and
 * width through the winning edge, which is recomputed.  A ray whose kind / idx is not a hit of its row is skipped, not
 * multiplied by 0.  No atomics: two calls give bit-identical gradients. */
int tds_range_scan_bwd(const tds_map_t* const* maps, int32_t n_maps, const int32_t* d_env_map, const float* d_absolute,
                       const int64_t* d_kind, const int64_t* d_idx, const float* d_grad_dist, int32_t B, int32_t A,
                       int32_t N, int32_t R, float* d_grad_absolute, void* stream);

/* ------------------------------------------------------------------------------------------
 * Time to collision (TTC; no counterpart in the reference): the first contact of every origin agent with any other
 * present agent under constant velocity, all pairs.
 * Inputs: d_state [B,N,4] (x, y, psi, v), d_size [B,N,2] (length, width), d_present [B,N] uint8 (0 / non-0);
 * n_agents = A <= N: rows 0..A-1 are the origins, all N rows are candidates (NPCs take part, as in compute_collision);
 * horizon H in seconds, finite and > 0.
 * Every agent keeps its heading and its speed: box j at time t has centre (x_j + t vx_j, y_j + t vy_j), with
 * vx_j = v_j c_j, vy_j = v_j s_j and (s_j, c_j) = sincos_cr(psi_j) (double precision, rounded), the heading evaluation
 * the whole path uses.  This is a definition, not the kinematic model's prediction: the bicycle's slip angle is ignored.
 * Pair (i, j), j != i with both present, float32, every operation rounded on its own (-fmad=false), IEEE division.
 * The four separating axes, in this order: 1. u_i = (c_i, s_i), 2. u_i⊥ = (-s_i, c_i), 3. u_j, 4. u_j⊥.
 * For axis n = (nx, ny): d0 = nx (x_j - x_i) + ny (y_j - y_i), s = nx (vx_j - vx_i) + ny (vy_j - vy_i), R = h_i + h_j.
 * A box's half-extent on its own axes is exactly 0.5 length or 0.5 width; on the other box's axes it is
 * |n·u| 0.5 length + |n·u⊥| 0.5 width (n·u = nx ux + ny uy).
 * Entry and exit per axis: s != 0: ta = (-R - d0) / s, tb = (R - d0) / s, entry min(ta, tb), exit max(ta, tb);
 * s == 0: entry -inf and exit +inf when |d0| <= R, otherwise the pair never touches.
 * T_in = max of the four entries, T_out = min of the four exits.  The pair touches within the horizon iff
 * max(T_in, 0) <= min(T_out, H); its time is T_in > 0 ? T_in : +0.0f (no negative zero: keys order by their bits).
 * Boxes that overlap at t = 0 give 0.  A pair whose time is NaN (a NaN entry or exit) never counts.
 * Outputs: d_ttc [B,A] float32 and d_idx [B,A] int64, the minimum over j of the pair time, ties to the smaller j (the
 * key is bits(t) << 32 | j).  No pair touches, or origin i is absent: ttc = +inf, idx = -1.
 * No host synchronisation, no allocation. */
int tds_time_to_collision(const float* d_state, const float* d_size, const uint8_t* d_present, int32_t B, int32_t A,
                          int32_t N, float horizon, float* d_ttc, int64_t* d_idx, void* stream);
/* The gradient of ttc with respect to the (x, y, psi, v) and (length, width) of the origin and of agent idx, where
 * 0 < ttc < inf.  There ttc = -(d0 + sgn(s) R) / s on the first axis, in the order above, whose entry equals T_in:
 * dt/dd0 = -1/s, dt/dR = -1/|s|, dt/ds = -t/s, chained through d0, s and R to both agents (d|x|/dx = sgn(x), 0 at 0).
 * d_idx as the forward wrote it; the pair and its axis are recomputed from the inputs.  d_grad_ttc [B,A],
 * d_grad_state [B,N,4], d_grad_size [B,N,2]: every element is written.  A row whose recomputed time is 0 or whose idx
 * is -1 (or not another present agent) is skipped by a branch, so an inf or NaN upstream value there reaches no
 * gradient.  No atomics: two calls give bit-identical gradients. */
int tds_time_to_collision_bwd(const float* d_state, const float* d_size, const uint8_t* d_present, int32_t B,
                              int32_t A, int32_t N, float horizon, const float* d_grad_ttc, const int64_t* d_idx,
                              float* d_grad_state, float* d_grad_size, void* stream);

/* ------------------------------------------------------------------------------------------
 * Offroad.  Replaces offroad_infraction_loss (infractions.py:176-229) + point_to_mesh_distance_pt
 * (infractions.py:86-173): out[b,a] = sum over the 4 box corners of (d2 if d2 > threshold else 0),
 * d2 = min over ALL map faces of the reference's squared point-triangle distance; times present.
 * maps[d_env_map[b]] is the map of environment b (d_env_map NULL: map 0 for all).
 * d_face [B,A,4] int32 or NULL receives the argmin face per corner (for the backward); -1 for a corner with no
 * gradient that needed no search: absent, or settled by the map's distance bound (d2 <= threshold).  The environment
 * variable TDS_OFFROAD_TRIAGE=0 searches every corner (same d_out).
 * ---------------------------------------------------------------------------------------- */
int tds_offroad_fwd(const tds_map_t* const* maps, int32_t n_maps, const int32_t* d_env_map,
                    const float* d_state, const float* d_lenwid, const uint8_t* d_present,
                    int32_t B, int32_t A, float threshold, float* d_out, int32_t* d_face, void* stream);
/* d_grad_out [B,A] -> d_grad_state [B,A,4] (x,y,psi; v gets 0), d_grad_lenwid [B,A,2] or NULL */
int tds_offroad_bwd(const tds_map_t* const* maps, int32_t n_maps, const int32_t* d_env_map,
                    const float* d_state, const float* d_lenwid, const uint8_t* d_present,
                    int32_t B, int32_t A, float threshold, const int32_t* d_face, const float* d_grad_out,
                    float* d_grad_state, float* d_grad_lenwid, void* stream);

/* ------------------------------------------------------------------------------------------
 * Birdview raster.  Replaces BirdviewRGBMeshGenerator.generate (mesh.py:1053-1157) +
 * BirdviewRenderer.render_frame (rendering/base.py:167-204) + CV2Renderer.render_rgb_mesh
 * (rendering/cv2.py:27-70) with pixel-identical output (cv2.fillConvexPoly integer rule).
 * ---------------------------------------------------------------------------------------- */
typedef struct {
    int32_t n_classes;                              /* size of the tables below, <= TDS_MAX_CLASSES */
    uint8_t active[TDS_MAX_CLASSES];                /* 1: the class may occur and gets a draw pass */
    uint8_t rank[TDS_MAX_CLASSES];                  /* draw order, 0 first (= highest z level) */
    uint8_t rgb[TDS_MAX_CLASSES][3];                /* colour of the class, 0..255 */
    int32_t agent_type_class[TDS_MAX_AGENT_TYPES];  /* class of agent type index t */
    int32_t direction_class;                        /* class of the direction triangle, -1: none */
    int32_t tl_state_class[TDS_MAX_TL_STATES];      /* class of traffic-light state index s */
} tds_palette_t;

/* bytes of the per-step scratch buffer (world-space dynamic triangles of every environment, the work counters of the
 * persistent raster grid and a list of up to B * N cameras for its second pass); always > 0.  Calls with more than
 * B * N cameras allocate library-owned scratch on first use, which cannot happen inside a CUDA graph capture. */
int64_t tds_raster_workspace_bytes(int32_t B, int32_t N, int32_t L, int32_t R);

/* Renders Nc cameras per environment.
 *   d_cam_xy, d_cam_sc [B,Nc,2]  camera positions and (sin, cos) of the camera orientation
 *   d_agent_state [B,N,4], d_agent_size [B,N,2], d_agent_type [B,N] int32 (NULL: type 0)
 *   d_present [B,N] uint8, or [B,Nc,N] when present_per_camera != 0 (rendering_mask)
 *   d_tl_corners [B,L,4,2], d_tl_state [B,L] int32 (L may be 0)
 *   d_rect_corners [B,R,4,2], d_rect_class [B,R] int32: extra rectangles (stop / yield signs)
 *   d_cam_tris [B,Nc,Tc,3,2], d_cam_tri_class [B,Nc,Tc] int32 (< 0: skipped): world-space triangles seen by ONE
 *       camera each - the goal-waypoint discs of generate(waypoints=...), mesh.py:1120-1145 (Tc may be 0)
 *   scale = 2 / fov, res = H = W (square only, as the reference)
 *   d_out [B,Nc,3,res,res] float32 in [0,255]
 *   d_workspace: tds_raster_workspace_bytes(B,N,L,R) bytes, required even when N = L = R = 0 */
int tds_raster_birdview(const tds_map_t* const* maps, int32_t n_maps, const int32_t* d_env_map,
                        int32_t B, int32_t Nc, int32_t N,
                        const float* d_cam_xy, const float* d_cam_sc,
                        const float* d_agent_state, const float* d_agent_size, const int32_t* d_agent_type,
                        const uint8_t* d_present, int32_t present_per_camera,
                        const float* d_tl_corners, const int32_t* d_tl_state, int32_t L,
                        const float* d_rect_corners, const int32_t* d_rect_class, int32_t R,
                        const float* d_cam_tris, const int32_t* d_cam_tri_class, int32_t Tc,
                        const tds_palette_t* palette, float scale, int32_t res,
                        float* d_out, void* d_workspace, void* stream);

/* Same raster with per-camera agent colours and a choice of the image format.
 * d_agent_class [B,Nc,N] uint8 or NULL: palette class of the RECTANGLE of agent n as camera c sees it, instead of the
 * class of its type - generate(custom_agent_colors=...), mesh.py:1092-1099 (the host layer gives every distinct
 * colour a palette class with the draw rank of the agent's type; the direction triangle keeps its class).
 * Image formats (the pixel values are integers in [0,255] in the reference too,
 * rendering/cv2.py:50-67, so the narrow formats lose nothing; they exist for consumers behind PCIe):
 *   TDS_IMAGE_F32  d_out float32 [B,Nc,3,res,res]  - the reference's dtype and layout (tds_raster_birdview)
 *   TDS_IMAGE_U8   d_out uint8   [B,Nc,3,res,res]  - the same values as bytes (4x fewer bytes)
 *   TDS_IMAGE_RANK d_out uint8   [B,Nc,res,res]    - per pixel the draw rank of the top-most class, 0 = background,
 *                  k >= 1 = the k-th entry of tds_raster_rank_table (12x fewer bytes) */
#define TDS_IMAGE_F32 0
#define TDS_IMAGE_U8 1
#define TDS_IMAGE_RANK 2
int tds_raster_birdview_fmt(const tds_map_t* const* maps, int32_t n_maps, const int32_t* d_env_map,
                            int32_t B, int32_t Nc, int32_t N,
                            const float* d_cam_xy, const float* d_cam_sc,
                            const float* d_agent_state, const float* d_agent_size, const int32_t* d_agent_type,
                            const uint8_t* d_present, int32_t present_per_camera,
                            const float* d_tl_corners, const int32_t* d_tl_state, int32_t L,
                            const float* d_rect_corners, const int32_t* d_rect_class, int32_t R,
                            const float* d_cam_tris, const int32_t* d_cam_tri_class, int32_t Tc,
                            const tds_palette_t* palette, float scale, int32_t res,
                            const uint8_t* d_agent_class, int32_t image_format, void* d_out, void* d_workspace,
                            void* stream);
/* Host helper for TDS_IMAGE_RANK: h_rgb[k][0..2] = colour of draw rank k (k = 0: background, black), h_class[k] = palette
 * class of rank k (-1 for k = 0); returns the number of ranks including the background, <= TDS_MAX_CLASSES + 1. */
int32_t tds_raster_rank_table(const tds_palette_t* palette, uint8_t h_rgb[][3], int32_t* h_class);

/* Measurement hook: when both are non-NULL cudaEvent_t handles, the next tds_raster_birdview calls on
 * this thread record `start` / `stop` on their stream immediately around the raster kernel launch
 * (the dominant kernel), so a benchmark can time it in situ.  Pass NULLs to disable. */
void tds_raster_set_timing_events(void* start_event, void* stop_event);

#ifdef __cplusplus
}
#endif
#endif /* TDS_B200_H */
