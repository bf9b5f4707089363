// msv_types.cuh -- device constant block and the structure-of-arrays HBM state.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/masurv.h"

// Config-derived constants, computed once on the host (msv_create) with the
// same float32/double arithmetic the reference performs on its Python numbers
// (citations in msv_abi.cu), then passed to every kernel by value.
struct WallC { float px, py, qs, qc, ang; float fat[4]; };

struct DevConst {
  int N;                 // environments on this device, padded to blocks * epb (SoA stride)
  int epb;               // environments per thread block of k_step (block = epb * G threads)
  int n_real;            // environments the caller asked for
  int A, B0, H0;         // n_agents, n_boxes, n_heals at reset
  int S;                 // agent row width: 8 (+1 with teams)
  int teams, omniscient, gameover_mode, health, melee_damage, melee_cooldown;
  int box_ownership, box_randomized, box_health, healing, inv_slots;
  int zone_phases, zone_cooldown, zone_damage, n_zones, zone_centers_random;
  int lidar_n, auto_reset, grid_n;  // grid_n = grid_size^2
  int immunity_cooldown, battle_royale, b2_variant;
  int toi_max_count;     // a contact takes part in SolveTOI while toiCount <= this (b2_maxSubSteps, or one less under MSV_B2_SUBSTEPS_GE)
  float r_alive, r_dead, r_kill, r_death;
  float agent_r, heal_r, item_r, box_h;
  float inv_mass, inv_I, friction, dt, dt_ratio1, damp;
  float imp_par[3], imp_nor[3], imp_ang[3];
  float melee_range, box_item_offset, drop_radius, pickup_r, give_r, cam_k1, lidar_depth;
  float cone_v[4][2], cone_n[4][2];
  float wall_hx, wall_hy;
  WallC walls[4];
  float grid_px[64], grid_py[64];
  float zone_r32[MSV_MAX_ZONES];          // float32(radiuses[i]), 0 appended
  double floor_size;
  double zone_radiuses[MSV_MAX_ZONES];
  double zone_centers[MSV_MAX_ZONES][2];
  double box_avg_w, box_std_w, box_avg_h, box_std_h, box_min_w, box_min_h;
  double lidar_ang[MSV_MAX_LASERS];       // i*(fov/(n-1)) - fov/2, as Python doubles
  uint32_t seed_lo, seed_hi;
  uint32_t env_offset;       // global index of env 0 (Philox counter word 0); msv_create rejects ids >= 2^32
  int profile;           // debug: accumulate per-phase clock64() deltas into g_prof
  // Tile hand-off from k_step to the observation kernel (set per launch by the host, 0 = off): a k_step block
  // that has stored its environments appends its index to the completion queue DevState::tq; the observation
  // kernel, launched programmatically dependent on k_step, consumes the queue in order while k_step's slower
  // blocks are still running.  Entries are (ticket << 32 | block); slot = atomicAdd(tq_tail, 1) - tq_base.
  uint32_t tq_ticket, tq_base;
  uint32_t pdl_wait;     // k_step was launched programmatically dependent on the previous step's last kernel: wait for it before touching state
};

// All per-environment state, structure-of-arrays: every array is
// [slot][N] with the environment index fastest: the leader lanes of a warp's
// consecutive environments read consecutive float4/int4 words of a field.
struct DevState {
  float4* akin0;   // [AC][N]  x, y, angle, vx
  float4* akin1;   // [AC][N]  vy, omega, sleep_time, flags (int bits: 1 alive, 2 awake)
  float4* afat;    // [AC][N]  fat AABB
  int4* aint;      // [AC][N]  health, cause, cooldown, inventory (n | kind_k << (4+2k))
  float4* ainv;    // [AC][4][N]  hx, hy, owner (int bits), rehulled (int bits)   (cold)
  float4* box0;    // [BC][N]  x, y, hx, hy
  int4* box1;      // [BC][N]  health, flags (1 has_health, 2 rehulled), cause, owner
  int* boxseq;     // [BC][N]
  float4* item0;   // [BC][N]  x, y, hx, hy
  int2* item1;     // [BC][N]  owner, seq
  float2* heal;    // [HC][N]  x, y
  int* healseq;    // [HC][N]
  float4* pend0;   // [BC][N]  x, y, hx, hy       (cold)
  int* pend1;      // [BC][N]  owner
  float2* zonec;   // [MSV_MAX_ZONES][N]
  float4* zonecur; // [N] x, y, r, -
  int4* zoneint;   // [N] phase, t_cooldown, t_shrink, endgame
  int4* hdr0;      // [N] counts (nb | ni<<8 | nh<<16 | np<<24), steps, episode, body_seq
  int4* hdr1;      // [N] contact_seq, first_step, overflow events, new-fixture flag
  unsigned long long* pex;  // [PW][N] pair exists
  unsigned long long* ptc;  // [PW][N] pair touching
  unsigned long long* pen;  // [PW][N] pair enabled
  uint32_t* pseq;  // [P][N]                          (cold)
  float2* pimp;    // [P][N] normal, tangent impulse  (cold)
  float* sreward;  // [AC][N]
  int* skills;     // [AC][N]
  int4* smisc;     // [N] steps, heals_used, boxes_placed, episodes
  float* epret;    // [AC][N] running return of the current episode, per agent
  // Pre-drawn reset records (k_spare): everything BaseEnv.reset draws from the RNG for an env's NEXT episode --
  // spawn cells, box shapes, zone centres -- computed off the step's critical path; valid iff spare_ep[e] == episode + 1
  float* spare;    // [N][MSV_SPARE_W]
  int* spare_ep;   // [N]
  unsigned long long* obm;  // [N] others_mask bits (observer i sees agent j: bit i*AC+j)
  unsigned* omask;          // [AC][N] non-omniscient: per observer, seen heals (bits 0-15), boxes (16-23), box items (24-31)
  unsigned long long* tq;   // [N / epb] completion queue of the current step's k_step blocks (see DevConst::tq_ticket)
  unsigned* tq_tail;        // [2] entries appended since the handle was created (mod 2^32); observation blocks finished
};

// layout of a reset record: boxes (x, y, hx, hy), heals (x, y), agents (x, y), zone centres (x, y)
#define MSV_SP_BOX 0
#define MSV_SP_HEAL (4 * MSV_MAX_BOXES)
#define MSV_SP_AGENT (MSV_SP_HEAL + 2 * MSV_MAX_HEALS)
#define MSV_SP_ZONE (MSV_SP_AGENT + 2 * MSV_MAX_AGENTS)
#define MSV_SPARE_W (MSV_SP_ZONE + 2 * MSV_MAX_ZONES)

struct DevOut {
  float* agent;          // [N][A][S]
  float* others;         // [N][A][A-1][S]
  float* others_mask;    // [N][A][A-1]
  float* zone;           // [N][6]            (same for every observer)
  float* heals;          // [N][H][2]         (same for every observer)
  float* heals_mask;     // [N][A][H]
  float* heal_slot;      // [N][A]
  float* heal_slot_mask; // [N][A]
  float* boxes;          // [N][B][11]
  float* boxes_mask;     // [N][A][B]
  float* box_items;      // [N][B][10]
  float* box_items_mask; // [N][A][B]
  float* box_slot;       // [N][A][8]
  float* box_slot_mask;  // [N][A]
  float* lidar_frac;     // [N][A][L]
  int* lidar_hit;        // [N][A][L]
  float* rewards;        // [N][A]
  uint8_t* dones;        // [N]
  float* episode_return; // [N][A]  return of the episode that just ended (rows valid where dones)
  int* episode_length;   // [N]     its length in steps
  uint8_t* immune;       // [N]     Health.immune as driven by ImmunityPhase (semantics.py:652-674)
  uint8_t* br_over;      // [N]     BattleRoyale.over (semantics.py:31-46)
  uint8_t* br_results;   // [N][A]  BattleRoyale.results (valid where br_over)
};

// ---- observation writer (k_obs2) -----------------------------------------
// The observation keys in DevOut order (agent .. box_slot_mask): tensor base and floats per environment.
struct ObsKey { float* base; int chunk; };
#define MSV_OBS_KEYS 14
struct ObsTable { ObsKey keys[MSV_OBS_KEYS]; };
// keys 4-7 (heals ..) exist only with heals, keys 8-13 (boxes ..) only with boxes
__host__ __device__ inline bool obs_key_used(int k, int H, int B) { return !((k >= 4 && k <= 7 && H == 0) || (k >= 8 && B == 0)); }
