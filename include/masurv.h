/*
 * masurv.h -- C ABI of libmasurv.so, the B200-native batched simulator for the
 * masurvival step path.
 *
 * This is the drop-in boundary for the hot path named by BASELINE.json
 * `north_star`: the reference's pseudo-gym API
 *     MaSurvival.reset()  masurvival/envs/masurvival_env.py:59-74
 *     MaSurvival.step()   masurvival/envs/masurvival_env.py:76-90
 *     flush_stats()       masurvival/envs/masurvival_env.py:471-480
 * (which in the reference fans out to Simulation.step, simulation.py:233-242,
 * the semantics.py modules and pybox2d's b2World.Step) is replaced, for a batch
 * of N independent environments, by the entry points below.  The reference has
 * no FFI of its own (pure Python on pybox2d), so these are the symbols a
 * ctypes binding inside the reference would load; INTEGRATION.md shows it.
 *
 * Plain C: pointers, sizes, PODs.  No torch types, no C++ in the signatures.
 * Every call returns MSV_OK (0) or a negative msv_err; no exception crosses.
 */
#ifndef MASURV_H
#define MASURV_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSV_ABI_VERSION 3

/* Compile-time capacities (per environment). */
#define MSV_MAX_AGENTS 8
#define MSV_MAX_BOXES 8
#define MSV_MAX_HEALS 16
#define MSV_MAX_SLOTS 4
#define MSV_MAX_ZONES 8 /* len(radiuses)+1 */
#define MSV_N_WALLS 4
#define MSV_MAX_LASERS 32
#define MSV_MAX_AA_PAIRS (MSV_MAX_AGENTS * (MSV_MAX_AGENTS - 1) / 2)

typedef enum msv_err {
  MSV_OK = 0,
  MSV_ERR_INVALID = -1,   /* bad argument / config out of capacity */
  MSV_ERR_CUDA = -2,      /* CUDA runtime error, see msv_last_error */
  MSV_ERR_NO_DEVICE = -3, /* no CUDA device: there is no CPU fallback */
  MSV_ERR_NAME = -4,      /* unknown tensor name */
  MSV_ERR_ALLOC = -5
} msv_err;

/* Item kinds held in an inventory slot (semantics.py:165-246). */
#define MSV_ITEM_NONE 0
#define MSV_ITEM_HEAL 1 /* semantics.py:637-649 */
#define MSV_ITEM_BOX 2  /* semantics.py:818-836, 864-884 */

/* "cause" of the last health change (semantics.py:490-500). */
#define MSV_CAUSE_NONE (-1)      /* None: never modified, or healed */
#define MSV_CAUSE_TEAM0 100      /* TeamBadge(0/1), semantics.py:917-933 */
#define MSV_CAUSE_ZONE 200       /* the SafeZone module, semantics.py:766 */
/* 0..A-1 = the attacking agent's index (no teams). */

#define MSV_GAMEOVER_ALLDEAD 0
#define MSV_GAMEOVER_LASTALIVE 1

/*
 * Flat POD form of the reference's nested config dict
 * (masurvival_env.py:140-238).  Python numbers stay double where the
 * reference does arithmetic on them as Python floats before narrowing to
 * Box2D's float32.
 */
typedef struct msv_config {
  int32_t n_agents;        /* agents.n_agents            env:166-169 */
  int32_t n_boxes;         /* boxes.reset_spawns.n_boxes env:192-195 */
  int32_t n_heals;         /* heals.reset_spawns.n_items env:211-214 */
  int32_t teams;           /* teams.twoteams             env:170-172 */
  int32_t omniscient;      /* observation.omniscent      env:141-143 */
  int32_t gameover_mode;   /* gameover.mode              env:154-156 */
  int32_t grid_size;       /* spawn_grid.grid_size       env:158-161 */
  int32_t health;          /* health.health              env:181-183 */
  int32_t melee_damage;    /* melee.damage               env:184-190 */
  int32_t melee_cooldown;  /* melee.cooldown; <0 = ContinuousMelee (env:309-312) */
  int32_t box_ownership;   /* boxes.ownership            env:196 */
  int32_t box_randomized;  /* 'randomized_shape' in boxes env:362-366 */
  int32_t box_health;      /* boxes.health               env:208 */
  int32_t healing;         /* heals.heal.healing         env:215-217 */
  int32_t inv_slots;       /* inventory.slots            env:219-221 */
  int32_t zone_phases;     /* safe_zone.phases           env:231-237 */
  int32_t zone_cooldown;
  int32_t zone_damage;
  int32_t zone_n_radiuses; /* len(radiuses) (without the appended 0) */
  int32_t zone_centers_random; /* centers == 'random' */
  int32_t lidar_n;         /* Lidars extension (simulation.py:357-392); 0 = off */
  int32_t auto_reset;      /* vector-env extension: 0 off; 1 reset finished envs inside step();
                              2 same + keep the finished episode's last observation in the
                              "terminal_<key>" tensors (valid for envs whose done flag is set) */
  float r_alive, r_dead, r_kill, r_death; /* reward_scheme env:144-153 */
  double floor_size;       /* spawn_grid.floor_size */
  double agent_size;       /* agents.agent_size (diameter) */
  double cam_fov, cam_depth;         /* cameras env:173-176 */
  double motor_impulse[3];           /* motors.impulse env:177-180 */
  double melee_range;
  double box_size;                   /* boxes.reset_spawns.box_size */
  double box_avg_w, box_std_w, box_avg_h, box_std_h, box_min_w, box_min_h;
  double box_item_size, box_item_offset; /* boxes.item env:204-207 */
  double heal_item_size;
  double pickup_radius;    /* auto_pickup.shape = circle(r) env:222-224 */
  double give_radius;      /* give.shape = circle(r)        env:225-227 */
  double drop_radius;      /* death_drop.radius             env:228-230 */
  double zone_radiuses[MSV_MAX_ZONES];
  double zone_centers[MSV_MAX_ZONES][2]; /* used when !zone_centers_random */
  double lidar_fov, lidar_depth;
  /* ---- modules the reference ships but its env never instantiates (env:322,336) ---- */
  int32_t immunity_cooldown; /* ImmunityPhase(cooldown), semantics.py:652-674; <0 = module absent.
                                Health.immune is written by it and read by nothing (semantics.py:490-500),
                                so only the "immune" tensor changes */
  int32_t battle_royale;     /* BattleRoyale, semantics.py:31-46: "br_over"/"br_results" tensors */
  /* Box2D details that differ between 2.3.x builds (the real pybox2d cannot be run here, DESIGN.md
   * section 4): bit 0 = clamp damping v *= clamp(1 - h*d, 0, 1) instead of the Pade form
   * v *= 1/(1 + h*d); bit 1 = b2PolygonShape::Set weld tolerance (0.5*linearSlop)^2 instead of
   * 2.3.0's 0.5*linearSlop; bit 2 = SolveTOI gives up at toiCount >= b2_maxSubSteps instead of >. */
  int32_t b2_variant;
  /* Vector-env extension (the reference has no step limit): 0 = none; T > 0 ends an episode as
   * "truncated" once it has run T steps (msv_env_state.steps >= T) without ending on that step.
   * Adds the "truncated" tensor (uint8[num_envs]); auto_reset resets truncated envs like finished ones
   * (and auto_reset 2 keeps their last observation), auto_reset 0 only flags them (msv_reset_envs).
   * The observation hand-off is off (msv_tile_plan out[3] = 0).  Negative values are refused. */
  int32_t max_episode_steps;
  /* Layout of the observation outputs: MSV_OBS_DICT writes one tensor per key; MSV_OBS_FLAT writes one
   * float32 tensor "obs_flat" [num_envs][n_agents][D] whose row [e][i] is agent i's observation: the
   * concatenation, in the order agent, zone, others, others_mask, heals, heals_mask, heal_slot,
   * heal_slot_mask, boxes, boxes_mask, box_items, box_items_mask, box_slot, box_slot_mask, lidar_frac,
   * of every key the config has (the keys stored once per env repeated in every agent's row).  Every key
   * keeps its name and dict-mode shape as a strided view into it (msv_tensor_info reports the strides);
   * "lidar_hit" stays a tensor of its own.  Other values are refused. */
  int32_t obs_layout;
  int32_t reserved1;       /* must be 0 */
} msv_config;
#define MSV_OBS_DICT 0
#define MSV_OBS_FLAT 1
#define MSV_B2_CLAMP_DAMPING 1
#define MSV_B2_WELD_SQUARED 2
#define MSV_B2_SUBSTEPS_GE 4

/*
 * One contact-pair record.  A pair "exists" while the two bodies' fat AABBs
 * overlap (b2ContactManager); seq orders contacts the way Box2D's LIFO contact
 * lists would (larger = newer = earlier in the list).
 */
typedef struct msv_pair {
  int32_t seq;      /* 0 = no contact between the two bodies */
  int32_t flags;    /* bit0 touching, bit1 enabled */
  float normal_impulse, tangent_impulse; /* warm-start cache, manifold point 0 */
} msv_pair;
#define MSV_PAIR_TOUCHING 1
#define MSV_PAIR_ENABLED 2

typedef struct msv_box_shape {
  float hx, hy;
  int32_t rehulled; /* 0: b2PolygonShape::SetAsBox vertex order; 1: went through
                       copy_shape -> b2PolygonShape::Set (simulation.py:43-45) */
} msv_box_shape;

/*
 * Complete state of ONE environment, host-side AoS.  This is the parity
 * injection / checkpoint format used by msv_get_state / msv_set_state; the
 * device keeps the same information in structure-of-arrays form.
 * Lists (boxes, box_items, heals, pending) are in the reference's
 * `group.bodies` list order (append on spawn, stable compaction on despawn).
 */
typedef struct msv_env_state {
  /* ---- agents, by stable index (IndexBodies, simulation.py:256-268) ---- */
  int32_t alive[MSV_MAX_AGENTS];
  int32_t health[MSV_MAX_AGENTS];
  int32_t cause[MSV_MAX_AGENTS];
  int32_t cooldown[MSV_MAX_AGENTS]; /* Melee.cooldowns, 0 = absent */
  float x[MSV_MAX_AGENTS], y[MSV_MAX_AGENTS], angle[MSV_MAX_AGENTS];
  float vx[MSV_MAX_AGENTS], vy[MSV_MAX_AGENTS], omega[MSV_MAX_AGENTS];
  float sleep_time[MSV_MAX_AGENTS];
  int32_t awake[MSV_MAX_AGENTS];
  float fat[MSV_MAX_AGENTS][4]; /* broad-phase fat AABB lx,ly,ux,uy */
  int32_t inv_n[MSV_MAX_AGENTS];
  int32_t inv_kind[MSV_MAX_AGENTS][MSV_MAX_SLOTS];
  msv_box_shape inv_shape[MSV_MAX_AGENTS][MSV_MAX_SLOTS];
  int32_t inv_owner[MSV_MAX_AGENTS][MSV_MAX_SLOTS];
  /* ---- boxes (static polygons), list order ---- */
  int32_t n_boxes;
  float box_x[MSV_MAX_BOXES], box_y[MSV_MAX_BOXES];
  msv_box_shape box_shape[MSV_MAX_BOXES];
  int32_t box_health[MSV_MAX_BOXES]; /* valid iff box_has_health */
  int32_t box_has_health[MSV_MAX_BOXES]; /* Q9: set at next Health.post_step */
  int32_t box_cause[MSV_MAX_BOXES];
  int32_t box_owner[MSV_MAX_BOXES]; /* MSV_CAUSE_NONE = no vulnerability set */
  int32_t box_seq[MSV_MAX_BOXES];   /* body creation sequence number */
  /* ---- box items on the floor (sensor circles), list order ---- */
  int32_t n_items;
  float item_x[MSV_MAX_BOXES], item_y[MSV_MAX_BOXES];
  msv_box_shape item_shape[MSV_MAX_BOXES];
  int32_t item_owner[MSV_MAX_BOXES];
  int32_t item_seq[MSV_MAX_BOXES]; /* body creation sequence number */
  /* ---- heal items on the floor, list order ---- */
  int32_t n_heals;
  float heal_x[MSV_MAX_HEALS], heal_y[MSV_MAX_HEALS];
  int32_t heal_seq[MSV_MAX_HEALS];
  /* ---- Object.next_spawns: boxes that died last step (semantics.py:853-861) */
  int32_t n_pending;
  float pend_x[MSV_MAX_BOXES], pend_y[MSV_MAX_BOXES];
  msv_box_shape pend_shape[MSV_MAX_BOXES];
  int32_t pend_owner[MSV_MAX_BOXES];
  /* ---- SafeZone (semantics.py:704-811) ---- */
  float zone_cx[MSV_MAX_ZONES], zone_cy[MSV_MAX_ZONES]; /* centers per phase */
  int32_t zone_phase, zone_t_cooldown, zone_t_shrink, zone_endgame;
  float zone_cur_x, zone_cur_y, zone_cur_r;
  /* ---- contact pairs ---- */
  msv_pair pair_aa[MSV_MAX_AA_PAIRS];               /* (i<j): j*(j-1)/2 + i */
  msv_pair pair_ab[MSV_MAX_AGENTS][MSV_MAX_BOXES];  /* agent x box list pos */
  msv_pair pair_aw[MSV_MAX_AGENTS][MSV_N_WALLS];    /* agent x wall (W,N,E,S) */
  /* ---- counters ---- */
  int32_t first_step;  /* 1 until the first b2World::Step (inv_dt0 == 0) */
  int32_t steps;       /* env.steps, env:73,88 */
  int32_t episode;     /* resets so far (Philox counter) */
  int32_t body_seq;    /* next body creation sequence number */
  int32_t contact_seq; /* last contact sequence number handed out */
  /* ---- episode stats accumulators (env:471-508) ---- */
  float stat_reward[MSV_MAX_AGENTS];
  int32_t stat_kills[MSV_MAX_AGENTS];
  int32_t stat_steps, stat_heals_used, stat_boxes_placed;
  int32_t stat_episodes;  /* auto-resets since the last flush (vector-env extension) */
  /* ---- running return / length of the current episode (per-env view of env:483-508) ---- */
  float ep_return[MSV_MAX_AGENTS];
} msv_env_state;

/* Sum over envs of the reference's flush_stats() dict (env:471-480). */
typedef struct msv_stats {
  double reward[MSV_MAX_AGENTS]; /* teams: [0],[1] = first member of team */
  int64_t kills[MSV_MAX_AGENTS];
  int64_t steps, heals_used, boxes_placed;
  int64_t episodes; /* auto-resets completed since the last flush */
} msv_stats;

typedef struct msv_handle msv_handle;

/* DLPack is re-declared by the caller (dlpack.h); here it is opaque. */
struct DLManagedTensor;

int msv_abi_version(void);
/* sizeof() of the PODs above as the library was compiled (layout check for
 * bindings that mirror the structs). */
int64_t msv_sizeof_config(void);
int64_t msv_sizeof_env_state(void);
int64_t msv_sizeof_stats(void);

/* Fill `cfg` with the reference's class default, env:140-238 (1v1, A=2). */
int msv_default_config(msv_config* cfg);

/* Replaces MaSurvival.__init__ (env:293-389) for `num_envs` environments on
 * CUDA device `device`.  `env_offset` is the global index of env 0 (multi-GPU
 * sharding: rank r passes r*num_envs) and only keys the Philox streams. */
int msv_create(const msv_config* cfg, int32_t num_envs, int32_t device,
               uint64_t seed, int64_t env_offset, msv_handle** out);
/* Frees the handle.  Device memory that is still referenced by live DLPack
 * exports (msv_tensor) stays allocated until the last of them is deleted, so
 * a tensor that outlives its environment never dangles. */
int msv_destroy(msv_handle* h);

/* Replaces BaseEnv.reset (env:59-74) for every env; stream-ordered. */
int msv_reset(msv_handle* h, void* cuda_stream);

/* Reset the environments whose byte in mask_dev (device pointer, uint8[num_envs], nonzero = reset)
 * is set, as BaseEnv.reset (env:59-74) for each of them; stream-ordered.  A reset env starts its next
 * episode (the same Philox draws as an auto-reset), gets msv_reset's observation, and its rewards,
 * dones and truncated are zeroed; its episode_return / episode_length rows (the last FINISHED
 * episode) stay, and the interrupted episode is not counted in msv_stats.episodes.  Every other env's
 * state and outputs are left bit-identical.  No host synchronisation and no allocation: a step and a
 * reset_envs can be captured together in a CUDA graph. */
int msv_reset_envs(msv_handle* h, const uint8_t* mask_dev, void* cuda_stream);

/* Replaces BaseEnv.step (env:76-90).  actions_dev: device pointer,
 * uint8[num_envs][n_agents][6], MultiDiscrete([3,3,3,2,2,2]) (env:451).
 * Results land in the library-owned tensors (msv_tensor). */
int msv_step(msv_handle* h, const uint8_t* actions_dev, void* cuda_stream);

/* Same, but actions come from HOST memory and rewards/dones are copied back
 * to host buffers inside the call (the end-to-end path bench.py times).
 * rewards_host: float[num_envs][n_agents]; dones_host: uint8[num_envs].
 * The read-back runs on an internal stream as soon as the step kernel is done,
 * overlapped with the observation kernels; the call returns when both the host
 * buffers and the observation tensors are complete.  The host buffers should be
 * page-locked (cudaHostAlloc / torch pin_memory): with pageable memory the
 * copies are staged by the driver and do not overlap the kernels. */
int msv_step_host(msv_handle* h, const uint8_t* actions_host,
                  float* rewards_host, uint8_t* dones_host, void* cuda_stream);

/* The same step returning the OBSERVATIONS as well (env:84,90: the step's main
 * result).  obs_host receives msv_obs_host_bytes() bytes: every observation
 * tensor (and the lidar block) in the library's de-duplicated layout, tensor
 * `name` at byte offset msv_obs_host_offset(name) (its first element), with the
 * shape and strides msv_tensor_info reports (MSV_OBS_FLAT: the block is
 * [obs_flat | lidar_hit] and the keys are strided views into obs_flat).  One device->host copy on the internal stream after
 * the observation kernels. */
int msv_step_host_obs(msv_handle* h, const uint8_t* actions_host,
                      float* rewards_host, uint8_t* dones_host, void* obs_host,
                      void* cuda_stream);
/* Split form for callers that keep several handles in flight (double-buffered
 * env groups): _async enqueues copy-in, kernels and copy-out and returns;
 * _wait blocks (spinning on an event, no stream synchronize) until the host
 * buffers of the last _async call are complete.  The next step on the same
 * handle is ordered after the copy-out by the library.  obs_host may be NULL.
 * The actions go up on an internal upload stream (ordered after this handle's
 * previous step, before this one's step kernel), so with several handles driven
 * through one launch stream a group's upload overlaps the other groups' kernels;
 * actions_host must stay unchanged until the step kernel has consumed it
 * (msv_step_host_wait of this call is sufficient). */
int msv_step_host_async(msv_handle* h, const uint8_t* actions_host,
                        float* rewards_host, uint8_t* dones_host, void* obs_host,
                        void* cuda_stream);
int msv_step_host_wait(msv_handle* h);
int64_t msv_obs_host_bytes(msv_handle* h);
int64_t msv_obs_host_offset(msv_handle* h, const char* name); /* -1: unknown */

/* Zero-copy export of a library-owned device tensor as DLPack.  Names are the
 * reference's observation keys (env:391-447) plus "rewards", "dones",
 * "episode_return", "episode_length", "lidar_frac", "lidar_hit", and
 * "truncated" (uint8[num_envs], only with max_episode_steps > 0: 1 where the
 * step limit ended the episode on the last step and the game did not; the
 * episode_* rows are valid where dones | truncated).  With MSV_OBS_FLAT also
 * "obs_flat" (and "terminal_obs_flat" under auto_reset 2); the observation
 * keys are then strided views into it (the strides are part of the export).
 * The deleter only drops a refcount. */
int msv_tensor(msv_handle* h, const char* name, struct DLManagedTensor** out);

/* Raw view of the same tensors (for non-DLPack callers / tests); strides in elements. */
int msv_tensor_info(msv_handle* h, const char* name, void** dev_ptr,
                    int32_t* ndim, int64_t shape[4], int64_t strides[4],
                    int32_t* dtype_code /*0 f32, 1 u8, 2 i32*/);

/* Parity injection / checkpoint: host AoS <-> device SoA, envs
 * [first, first+count). Synchronous. */
int msv_get_state(msv_handle* h, int32_t first, int32_t count,
                  msv_env_state* out);
int msv_set_state(msv_handle* h, int32_t first, int32_t count,
                  const msv_env_state* in);

/* Recompute observations from the current state without stepping
 * (fetch_observations, env:510-657), e.g. after msv_set_state. */
int msv_observe(msv_handle* h, void* cuda_stream);

/* Top-down RGB picture of envs [first, first+count), out_dev: device pointer to
 * uint8[count][height][width][3] (row 0 at the top, +y up; the viewport is the
 * floor and its walls with a margin of a wall's width, centred on the origin).
 * Stream-ordered after everything already enqueued on cuda_stream (e.g. the
 * msv_step whose result it shows); reads the state, writes only out_dev.
 * height and width are 1..4096; MSV_RENDER_LIDAR needs lidars in the config.
 * Colours are the entries of msv_render_palette, in this order: background,
 * floor, floor outside the safe zone, zone ring, next-zone ring, wall, heal,
 * box item, box, agent 0 .. agent 7, team 0, team 1, heading tick, lidar ray. */
#define MSV_RENDER_LIDAR 1u   /* draw the lidar rays (only with lidars configured) */
int msv_render(msv_handle* h, int32_t first, int32_t count, int32_t height, int32_t width,
               uint32_t flags, uint8_t* out_dev, void* cuda_stream);
/* Copies min(capacity, n) colours (3 bytes each) to out_rgb and returns n, the
 * number of colours; out_rgb may be NULL when capacity is 0.  Needs no device. */
int msv_render_palette(uint8_t* out_rgb, int32_t capacity);

/* Global state for centralised critics: one float32 row of Ds floats per env,
 * what an omniscient observer sees, stored once, plus an alive mask and the
 * step count (no lidar).  Keys in this order; the heal keys exist only with
 * n_heals > 0, the box keys only with n_boxes > 0; masks: 0 present, 1 absent.
 *   agents [A][S]          obs['agent'][e] (id, (team), health, x, y, angle,
 *                          vx, vy, omega; a dead agent keeps id and team)
 *   agents_mask [A]        0 alive, 1 dead
 *   zone [6]               obs['zone'][e]
 *   heals [H][2], heals_mask [H]            0 where k < n_heals
 *   heal_slot [A], heal_slot_mask [A]       obs['heal_slot'][e, i, 0, 0] and its mask
 *   boxes [B][11], boxes_mask [B]           0 where k < n_boxes
 *   box_items [B][10], box_items_mask [B]   0 where k < n_items
 *   box_slot [A][8], box_slot_mask [A]      obs['box_slot'][e, i, 0] and its mask
 *   steps [1]              the episode's step count (msv_env_state.steps)
 * Ds = A*(S+1) + 6 + [H>0]*(3H + 2A) + [B>0]*(23B + 9A) + 1 (S = 8, 9 with teams).
 * Width Ds of the row for cfg (host only, no device), or MSV_ERR_INVALID. */
int msv_global_state_dim(const msv_config* cfg);
/* Turn on the "global_state" output (float32 [num_envs][Ds]; with auto_reset 2
 * also "terminal_global_state", rows valid where the episode finished on the
 * last step, the other rows untouched).  Allocates the buffers, writes the row
 * of every env for the current state on cuda_stream, and from then on every
 * call that writes observations (step, reset, reset_envs, observe, the
 * step_host forms) writes it too, after the observation kernels.  Each key is
 * also exported as a strided view "global_state_<key>" (and
 * "terminal_global_state_<key>"): shape [num_envs][key shape], stride Ds
 * between envs; before the call these names are unknown (MSV_ERR_NAME).
 * Idempotent (a second call rewrites the rows; pointers are unchanged).
 * Refused (MSV_ERR_INVALID) for a NULL handle or while cuda_stream is being
 * captured (it allocates).  The row is not part of the host read-back. */
int msv_enable_global_state(msv_handle* h, void* cuda_stream);

/* flush_stats (env:471-480) summed over all envs; zeroes the accumulators.
 * Synchronises the device first (work queued on any stream is complete). */
int msv_flush_stats(msv_handle* h, msv_stats* out);

/* Algorithmic HBM bytes one msv_step moves per env (state read+write,
 * actions, observations, rewards, dones) -- the roofline numerator -- and
 * its split by kernel (which: 0 step kernel, 1 observation gather, 2 lidar,
 * 3 global state: 0 until msv_enable_global_state). */
int64_t msv_bytes_per_env_step(msv_handle* h);
int64_t msv_kernel_bytes_per_env(msv_handle* h, int32_t which);
/* The part of it written by the observation kernel (k_obs2). */
int64_t msv_obs_bytes_per_env(msv_handle* h);
int64_t msv_kernel_launches(msv_handle* h); /* launches since create */
/* How the batch is tiled onto the GPU: out[0] environments per thread block of
 * the step kernel, out[1] its blocks, out[2] its threads per block, out[3] 1 when
 * the observation kernels are launched programmatically dependent on the step
 * kernel and consume its tiles as they finish (not with auto_reset 2 or a step
 * limit, whose steps run more kernels in between; the vectorised counterpart of
 * env:76-90 has no analogue in the reference: it steps one env at a time). */
int msv_tile_plan(msv_handle* h, int32_t out[4]);
/* The planner behind it, without a device (pure host logic): how num_envs
 * environments of cfg would be tiled onto a GPU with sm_count SMs and
 * smem_per_block bytes of opt-in shared memory per block (B200: 148, 232448).
 * out = {envs per block, blocks, threads per block, capacity class 0..2}. */
int msv_plan_tile(const msv_config* cfg, int32_t num_envs, int32_t sm_count,
                  int64_t smem_per_block, int32_t out[4]);
int64_t msv_device_bytes(msv_handle* h);    /* HBM allocated by the handle */

const char* msv_last_error(msv_handle* h);

/* Philox4x32-10 draw exposed for tests: counter (c0..c3), key (k0,k1). */
void msv_philox4x32(const uint32_t ctr[4], const uint32_t key[2],
                    uint32_t out[4]);

#ifdef __cplusplus
}
#endif
#endif /* MASURV_H */
