// msv_abi.cu -- the C ABI of libmasurv.so (include/masurv.h): handle life
// cycle, config -> device constants, SoA allocation, AoS<->SoA state
// exchange, DLPack export, launches.  There is NO CPU fallback: every entry
// point that computes fails with MSV_ERR_NO_DEVICE when no CUDA device exists.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>
#include <map>

#include "../../include/masurv.h"
#include "msv_launch.h"

// ---- minimal DLPack (dlpack.h v0.8 layout) --------------------------------
extern "C" {
typedef struct { int32_t device_type; int32_t device_id; } DLDevice;
typedef struct { uint8_t code; uint8_t bits; uint16_t lanes; } DLDataType;
typedef struct {
  void* data; DLDevice device; int32_t ndim; DLDataType dtype;
  int64_t* shape; int64_t* strides; uint64_t byte_offset;
} DLTensor;
typedef struct DLManagedTensor {
  DLTensor dl_tensor; void* manager_ctx; void (*deleter)(struct DLManagedTensor*);
} DLManagedTensor;
}

struct TensorInfo { void* ptr; int ndim; int64_t shape[4]; int dtype; /*0 f32, 1 u8, 2 i32*/ };

struct msv_handle {
  msv_config cfg;
  DevConst C;
  DevState S;
  DevOut O;
  int cap, AC, BC, HC, P, PW, sm_words;
  int device;
  std::vector<void*> allocs;
  std::map<std::string, TensorInfo> tensors;
  uint8_t* d_actions;       // staging for msv_step_host
  // msv_step_host* read rewards/dones back on a second stream as soon as the step kernel is done
  // (overlapping the copy with the observation kernels) and the observation arena after them
  cudaStream_t copy_stream = nullptr; cudaEvent_t ev_step = nullptr, ev_obs = nullptr, ev_copy = nullptr;
  // msv_step_host*: the actions go up on a stream of their own, so that with several handles driven through one
  // launch stream (env groups in flight) a group's upload overlaps the other groups' kernels instead of sitting
  // in stream order in front of its own step kernel
  cudaStream_t up_stream = nullptr; cudaEvent_t ev_up = nullptr, ev_done = nullptr; bool done_valid = false;
  float* host_rewards = nullptr; uint8_t* host_dones = nullptr; void* host_obs = nullptr;   // destinations of the pending read-back (one step)
  bool copy_pending = false;     // ev_copy was recorded and nobody waited for it yet
  // every output tensor lives in ONE device arena: [rewards | dones | observation keys | lidar]
  char* arena = nullptr; size_t arena_bytes = 0, obs_begin = 0, obs_end = 0;
  size_t device_bytes = 0;
  bool zombie = false;           // msv_destroy was called while DLPack exports were alive
  // k_spare (pre-drawn reset records) runs on a side stream beside the observation kernels and is joined
  // back into the caller's stream before msv_step returns (fork/join inside the call: graph-capture safe)
  cudaStream_t side_stream = nullptr; cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  uint32_t tq_ticket = 0, tq_base = 0; bool handoff = true;   // k_step -> k_obs2 tile hand-off (MSV_NO_HANDOFF=1 turns it off)
  bool last_was_step = false; cudaStream_t last_stream = nullptr;   // the last call on last_stream ended with the hand-off's observation kernel: the next k_step is programmatically dependent on it
  // debug: CUDA-event timing of the kernels of msv_step (bench.py's roofline numerator)
  bool timing = false; std::vector<cudaEvent_t> tev; size_t tev_used = 0;
  double* d_stat_reward; unsigned long long* d_stat_kills; unsigned long long* d_stat_misc;
  int64_t launches;
  ObsTable obs;
  int64_t obs_floats = 0;    // floats of one environment's observation keys (the keys the config has)
  ObsTable obs_term;         // auto_reset == 2: same table, writing the "terminal_<key>" tensors
  DevOut O_term;             // auto_reset == 2: O with the lidar pointers on the "terminal_lidar_*" tensors
  uint8_t* truncated = nullptr;   // max_episode_steps > 0: the "truncated" tensor [N]
  uint8_t* finished = nullptr;    // max_episode_steps > 0: dones | truncated of the last step [N] (k_truncate)
  int64_t exported;          // live DLPack exports
  std::string err;
};

#define CK(call)                                                                      \
  do {                                                                                \
    cudaError_t _e = (call);                                                          \
    if (_e != cudaSuccess) {                                                          \
      h->err = std::string(#call) + ": " + cudaGetErrorString(_e);                   \
      return MSV_ERR_CUDA;                                                            \
    }                                                                                 \
  } while (0)

static thread_local std::string g_err;

// the calling thread's current device is restored when a DevGuard goes out of scope
struct DevGuard {
  int prev = -1; bool switched = false;
  explicit DevGuard(int dev) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) switched = cudaSetDevice(dev) == cudaSuccess;
  }
  ~DevGuard() { if (switched) cudaSetDevice(prev); }
};


// ---- host float32 helpers (same arithmetic as the reference's pybox2d calls)
static void h_rot(float angle, float* s, float* c) { *s = (float)sin((double)angle); *c = (float)cos((double)angle); }
// sim.from_polar (simulation.py:20-23)
static void h_from_polar(double length, double angle, float out[2]) {
  float s, c; h_rot((float)angle, &s, &c);
  float L = (float)length;
  out[0] = c * L + (-s) * 0.0f; out[1] = s * L + c * 0.0f;
}
// b2PolygonShape::Set for the 4-vertex camera cone (simulation.py:321-328)
static void h_polygon_set4(const float vin[4][2], float vout[4][2], float nout[4][2]) {
  int n = 4, i0 = 0; float x0 = vin[0][0];
  for (int i = 1; i < n; ++i) {
    float x = vin[i][0];
    if (x > x0 || (x == x0 && vin[i][1] < vin[i0][1])) { i0 = i; x0 = x; }
  }
  int hull[8], m = 0, ih = i0;
  for (;;) {
    hull[m] = ih;
    int ie = 0;
    for (int j = 1; j < n; ++j) {
      if (ie == ih) { ie = j; continue; }
      float rx = vin[ie][0] - vin[hull[m]][0], ry = vin[ie][1] - vin[hull[m]][1];
      float vx = vin[j][0] - vin[hull[m]][0], vy = vin[j][1] - vin[hull[m]][1];
      float c = rx * vy - ry * vx;
      if (c < 0.0f) ie = j;
      if (c == 0.0f && vx * vx + vy * vy > rx * rx + ry * ry) ie = j;
    }
    ++m; ih = ie;
    if (ie == i0 || m >= 4) break;
  }
  for (int i = 0; i < 4; ++i) { int k = i < m ? i : m - 1; vout[i][0] = vin[hull[k]][0]; vout[i][1] = vin[hull[k]][1]; }
  for (int i = 0; i < 4; ++i) {
    int i2 = i + 1 < 4 ? i + 1 : 0;
    float ex = vout[i2][0] - vout[i][0], ey = vout[i2][1] - vout[i][1];
    float nx = 1.0f * ey, ny = -1.0f * ex;
    float len = sqrtf(nx * nx + ny * ny);
    if (!(len < 1.1920929e-7f)) { float inv = 1.0f / len; nx *= inv; ny *= inv; }
    nout[i][0] = nx; nout[i][1] = ny;
  }
}

static int build_const(const msv_config* c, int N, uint64_t seed, int64_t env_offset, DevConst* D) {
  memset(D, 0, sizeof *D);
  D->N = N; D->epb = 0; D->n_real = N;   /* N (the padded SoA stride) and epb are set by plan_blocks() */ D->A = c->n_agents; D->B0 = c->n_boxes; D->H0 = c->n_heals;
  D->S = 8 + (c->teams ? 1 : 0);
  D->teams = c->teams; D->omniscient = c->omniscient; D->gameover_mode = c->gameover_mode;
  D->health = c->health; D->melee_damage = c->melee_damage; D->melee_cooldown = c->melee_cooldown;
  D->box_ownership = c->box_ownership; D->box_randomized = c->box_randomized; D->box_health = c->box_health;
  D->healing = c->healing; D->inv_slots = c->inv_slots;
  D->zone_phases = c->zone_phases; D->zone_cooldown = c->zone_cooldown; D->zone_damage = c->zone_damage;
  D->n_zones = c->zone_n_radiuses + 1; D->zone_centers_random = c->zone_centers_random;
  D->lidar_n = c->lidar_n; D->auto_reset = c->auto_reset; D->grid_n = c->grid_size * c->grid_size;
  D->immunity_cooldown = c->immunity_cooldown; D->battle_royale = c->battle_royale; D->b2_variant = c->b2_variant;
  D->toi_max_count = (c->b2_variant & MSV_B2_SUBSTEPS_GE) ? 7 : 8;   // b2_maxSubSteps = 8: "toiCount > 8" vs "toiCount >= 8" skips the contact
  D->r_alive = c->r_alive; D->r_dead = c->r_dead; D->r_kill = c->r_kill; D->r_death = c->r_death;
  D->agent_r = (float)(c->agent_size / 2);          // semantics.py:16-18
  D->heal_r = (float)(c->heal_item_size / 2);       // semantics.py:24-25
  D->item_r = (float)(c->box_item_size / 2);
  D->box_h = (float)(c->box_size / 2.);             // semantics.py:20-22
  {  // b2CircleShape::ComputeMass + b2Body::ResetMassData, density 1
    const float b2_pi = 3.14159265359f;
    float r = D->agent_r, density = 1.0f;
    float mass = density * b2_pi * r * r;
    float I = mass * (0.5f * r * r + 0.0f);
    D->inv_mass = 1.0f / mass;
    I -= mass * 0.0f;
    D->inv_I = 1.0f / I;
  }
  D->friction = sqrtf(0.2f * 0.2f);                  // b2MixFriction of the fixture default
  D->dt = (float)(1.0 / 60);                         // simulation.py:219
  D->dt_ratio1 = (1.0f / D->dt) * D->dt;
  D->damp = 1.0f / (1.0f + D->dt * (float)0.8);      // simulation.py:118, Pade damping (b2Island::Solve, Box2D >= 2.3.0)
  if (c->b2_variant & MSV_B2_CLAMP_DAMPING) {        // Box2D <= 2.2: v *= b2Clamp(1 - h * damping, 0, 1)
    float d = 1.0f - D->dt * (float)0.8;
    D->damp = d < 0.0f ? 0.0f : (d > 1.0f ? 1.0f : d);
  }
  static const double dtab[3] = {-1., 0., 1.};       // env:742
  for (int a = 0; a < 3; ++a) {
    D->imp_par[a] = (float)(dtab[a] * c->motor_impulse[0]);
    D->imp_nor[a] = (float)(dtab[a] * c->motor_impulse[1]);
    D->imp_ang[a] = (float)(dtab[a] * c->motor_impulse[2]);
  }
  D->melee_range = (float)c->melee_range; D->box_item_offset = (float)c->box_item_offset;
  D->drop_radius = (float)c->drop_radius; D->pickup_r = (float)c->pickup_radius; D->give_r = (float)c->give_radius;
  D->cam_k1 = (float)(1 + 1e-6);                     // simulation.py:349
  D->lidar_depth = (float)c->lidar_depth;
  {
    float vin[4][2] = {{0.0f, 0.0f}, {0, 0}, {(float)c->cam_depth, 0.0f}, {0, 0}};
    h_from_polar(c->cam_depth, +c->cam_fov / 2, vin[1]);
    h_from_polar(c->cam_depth, -c->cam_fov / 2, vin[3]);
    h_polygon_set4(vin, D->cone_v, D->cone_n);
  }
  {  // ThickRoomWalls, semantics.py:685-695
    double height = c->floor_size, width = height / 100;
    D->wall_hx = (float)(width / 2.); D->wall_hy = (float)(height / 2.);
    float o = (float)(c->floor_size / 2), hp = (float)(M_PI / 2);
    float wx[4] = {-o, 0.0f, o, 0.0f}, wy[4] = {0.0f, o, 0.0f, -o}, wa[4] = {0.0f, hp, 0.0f, hp};
    for (int k = 0; k < 4; ++k) {
      WallC& w = D->walls[k];
      w.px = wx[k]; w.py = wy[k]; w.ang = wa[k]; h_rot(wa[k], &w.qs, &w.qc);
      float hx = D->wall_hx, hy = D->wall_hy;
      float vs[4][2] = {{-hx, -hy}, {hx, -hy}, {hx, hy}, {-hx, hy}};
      float lx = 0, ly = 0, ux = 0, uy = 0;
      for (int v = 0; v < 4; ++v) {
        float x = (w.qc * vs[v][0] - w.qs * vs[v][1]) + w.px, y = (w.qs * vs[v][0] + w.qc * vs[v][1]) + w.py;
        if (v == 0) { lx = ux = x; ly = uy = y; }
        else { lx = x < lx ? x : lx; ly = y < ly ? y : ly; ux = x > ux ? x : ux; uy = y > uy ? y : uy; }
      }
      const float pr = 2.0f * 0.005f, ext = 0.1f;
      w.fat[0] = (lx - pr) - ext; w.fat[1] = (ly - pr) - ext; w.fat[2] = (ux + pr) + ext; w.fat[3] = (uy + pr) + ext;
    }
  }
  {  // square_grid, semantics.py:987-992
    int g = c->grid_size;
    for (int k = 0; k < g * g; ++k) {
      int i = k % g, j = k / g;
      double ci = (double)i / g + 0.5 / g, cj = (double)j / g + 0.5 / g;
      D->grid_px[k] = (float)(c->floor_size * ci - c->floor_size / 2.);
      D->grid_py[k] = (float)(c->floor_size * cj - c->floor_size / 2.);
    }
  }
  for (int z = 0; z < MSV_MAX_ZONES; ++z) {
    double r = z < c->zone_n_radiuses ? c->zone_radiuses[z] : 0.0;   // semantics.py:726-727
    D->zone_radiuses[z] = r; D->zone_r32[z] = (float)r;
    if (z < c->zone_n_radiuses) { D->zone_centers[z][0] = c->zone_centers[z][0]; D->zone_centers[z][1] = c->zone_centers[z][1]; }
  }
  D->floor_size = c->floor_size;
  D->box_avg_w = c->box_avg_w; D->box_std_w = c->box_std_w; D->box_avg_h = c->box_avg_h; D->box_std_h = c->box_std_h;
  D->box_min_w = c->box_min_w; D->box_min_h = c->box_min_h;
  for (int r = 0; r < c->lidar_n && r < MSV_MAX_LASERS; ++r)     // simulation.py:385-392
    D->lidar_ang[r] = c->lidar_n > 1 ? r * (c->lidar_fov / (c->lidar_n - 1)) - c->lidar_fov / 2. : 0.0;
  D->seed_lo = (uint32_t)seed; D->seed_hi = (uint32_t)(seed >> 32);
  D->env_offset = (uint32_t)env_offset;
  return 0;
}

// Tile size of k_step: a block is a tile of `epb` environments (epb * G threads, G = agent capacity = lanes per
// environment).  A block's warps run the step in phase lock-step (block barriers between the phases) and so share
// one pass over its ~560 KB of instructions; two blocks on an SM sit in different phases and evict each other's
// lines from the instruction caches.  Measured on the stationary 2v2 workload (16 384 envs, profiles/r02_tiles.txt):
// two 64-env blocks of 256 threads per SM 124.9 us/step; ONE block of 512 threads per SM with 128 envs 112.5,
// 120 envs 113.0, 112 envs (147 blocks: every SM busy) 109.8.  So: one block per SM, as few waves as the block
// capacity allows; a batch that fits one wave is spread over every SM (a block lasts as long as its slowest
// environment in every phase, so smaller tiles shorten every block), a batch that needs several waves takes the
// largest tile (blocks are handed out as SMs free up; ffa + lidar, 32 768 envs: 64-env tiles 1 239 us, 56 -- four
// even waves -- 1 288, 48: 1 327).
static long plan_tile(int G, int sm_words, long n, long sms, size_t smem_blk_max) {
  const long wpe = 32 / G;
  long cap = MSV_TPB / G;                                          // by threads (128 registers each: 512 fill the register file)
  const long by_smem = (long)(smem_blk_max / ((size_t)sm_words * sizeof(float)));
  if (by_smem < cap) cap = by_smem;
  cap = cap / wpe * wpe; if (cap < wpe) cap = wpe;
  if (sms < 1) sms = 1;
  if (n < 1) n = 1;
  const long waves = (n + cap * sms - 1) / (cap * sms);
  long best = (n + sms - 1) / sms;                                  // one wave: spread the batch over every SM
  best = (best + wpe - 1) / wpe * wpe;
  if (waves > 1) best = cap;
  if (best > cap) best = cap;
  if (best < wpe) best = wpe;
  return best;
}
static int capacity_class(const msv_config* cfg) {
  return (cfg->n_agents <= 2 && cfg->n_boxes <= 4 && cfg->n_heals <= 4) ? 0
       : (cfg->n_agents <= 4 && cfg->n_boxes <= 4 && cfg->n_heals <= 4) ? 1 : 2;
}
static void plan_blocks(msv_handle* h, int device) {
  cudaDeviceProp pr; int sms = 148; size_t smem_blk_max = 227 * 1024;
  if (cudaGetDeviceProperties(&pr, device) == cudaSuccess) { sms = pr.multiProcessorCount; smem_blk_max = pr.sharedMemPerBlockOptin; }
  const int G = h->AC, wpe = 32 / G, n = h->C.n_real;
  long best = plan_tile(G, h->sm_words, n, sms, smem_blk_max);
  if (const char* ov = getenv("MSV_EPB")) {                         // development override
    const long cap = plan_tile(G, h->sm_words, (long)1 << 40, 1, smem_blk_max);   // (many waves -> the capacity)
    int v = atoi(ov); if (v >= wpe && v <= cap && v % wpe == 0) best = v;
  }
  h->C.epb = (int)best;
  h->C.N = (int)((n + best - 1) / best * best);
}
/* The same planner without a device (host logic only): how `num_envs` environments of `cfg` would be tiled onto a
 * GPU with `sm_count` SMs and `smem_per_block` bytes of opt-in shared memory per block.
 * out = {envs per block, blocks, threads per block, capacity class}. */
int msv_plan_tile(const msv_config* cfg, int32_t num_envs, int32_t sm_count, int64_t smem_per_block, int32_t out[4]) {
  if (!cfg || !out || num_envs < 1 || sm_count < 1 || smem_per_block < 1024) return MSV_ERR_INVALID;
  const int cap = capacity_class(cfg);
  int AC, BC, HC, P, PW, smw;
  msv_capacity(cap, &AC, &BC, &HC, &P, &PW, &smw);
  const long epb = plan_tile(AC, smw, num_envs, sm_count, (size_t)smem_per_block);
  out[0] = (int32_t)epb; out[1] = (int32_t)((num_envs + epb - 1) / epb); out[2] = (int32_t)(epb * AC); out[3] = cap;
  return MSV_OK;
}

template <typename T> static int dalloc(msv_handle* h, T** p, size_t count) {
  void* q = nullptr;
  size_t bytes = (count ? count : 1) * sizeof(T);
  cudaError_t e = cudaMalloc(&q, bytes);
  if (e != cudaSuccess) { h->err = std::string("cudaMalloc: ") + cudaGetErrorString(e); return MSV_ERR_ALLOC; }
  cudaMemset(q, 0, bytes);
  h->allocs.push_back(q);
  h->device_bytes += bytes;
  *p = (T*)q;
  return 0;
}

static void reg(msv_handle* h, const char* name, void* ptr, int dtype, std::initializer_list<int64_t> shape) {
  TensorInfo t; t.ptr = ptr; t.ndim = (int)shape.size(); t.dtype = dtype;
  int i = 0; for (auto s : shape) t.shape[i++] = s;
  h->tensors[name] = t;
}

// ---- AoS <-> SoA -----------------------------------------------------------
struct Mirror {
  std::vector<float4> akin0, akin1, afat, ainv, box0, item0, pend0, zonecur;
  std::vector<int4> aint, box1, zoneint, hdr0, hdr1, smisc;
  std::vector<int> boxseq, healseq, pend1, skills;
  std::vector<int2> item1;
  std::vector<float2> heal, zonec, pimp;
  std::vector<unsigned long long> pex, ptc, pen;
  std::vector<uint32_t> pseq;
  std::vector<float> sreward, epret;
};
// Only the columns [first, first+count) of every [slots][N] array cross the bus: the mirror's
// arrays are [slots][count] (a checkpoint of k envs costs O(k), not O(N)).
struct Slice { size_t first, count, N; };
template <typename T> static cudaError_t dl(std::vector<T>& v, const T* d, size_t slots, const Slice& sl) {
  v.resize(slots * sl.count);
  return cudaMemcpy2D(v.data(), sl.count * sizeof(T), d + sl.first, sl.N * sizeof(T), sl.count * sizeof(T), slots, cudaMemcpyDeviceToHost);
}
template <typename T> static cudaError_t ul(const std::vector<T>& v, T* d, const Slice& sl) {
  const size_t slots = v.size() / sl.count;
  return cudaMemcpy2D(d + sl.first, sl.N * sizeof(T), v.data(), sl.count * sizeof(T), sl.count * sizeof(T), slots, cudaMemcpyHostToDevice);
}
static int download(msv_handle* h, Mirror& m, const Slice& sl) {
  const size_t AC = h->AC, BC = h->BC, HC = h->HC, P = h->P, PW = h->PW;
  DevState& S = h->S;
  CK(cudaDeviceSynchronize());
  CK(dl(m.akin0, S.akin0, AC, sl)); CK(dl(m.akin1, S.akin1, AC, sl)); CK(dl(m.afat, S.afat, AC, sl));
  CK(dl(m.aint, S.aint, AC, sl)); CK(dl(m.ainv, S.ainv, AC * 4, sl));
  CK(dl(m.box0, S.box0, BC, sl)); CK(dl(m.box1, S.box1, BC, sl)); CK(dl(m.boxseq, S.boxseq, BC, sl));
  CK(dl(m.item0, S.item0, BC, sl)); CK(dl(m.item1, S.item1, BC, sl));
  CK(dl(m.heal, S.heal, HC, sl)); CK(dl(m.healseq, S.healseq, HC, sl));
  CK(dl(m.pend0, S.pend0, BC, sl)); CK(dl(m.pend1, S.pend1, BC, sl));
  CK(dl(m.zonec, S.zonec, (size_t)MSV_MAX_ZONES, sl)); CK(dl(m.zonecur, S.zonecur, 1, sl)); CK(dl(m.zoneint, S.zoneint, 1, sl));
  CK(dl(m.hdr0, S.hdr0, 1, sl)); CK(dl(m.hdr1, S.hdr1, 1, sl));
  CK(dl(m.pex, S.pex, PW, sl)); CK(dl(m.ptc, S.ptc, PW, sl)); CK(dl(m.pen, S.pen, PW, sl));
  CK(dl(m.pseq, S.pseq, P, sl)); CK(dl(m.pimp, S.pimp, P, sl));
  CK(dl(m.sreward, S.sreward, AC, sl)); CK(dl(m.skills, S.skills, AC, sl)); CK(dl(m.smisc, S.smisc, 1, sl));
  CK(dl(m.epret, S.epret, AC, sl));
  return MSV_OK;
}
static int upload(msv_handle* h, const Mirror& m, const Slice& sl) {
  DevState& S = h->S;
  CK(ul(m.akin0, S.akin0, sl)); CK(ul(m.akin1, S.akin1, sl)); CK(ul(m.afat, S.afat, sl)); CK(ul(m.aint, S.aint, sl)); CK(ul(m.ainv, S.ainv, sl));
  CK(ul(m.box0, S.box0, sl)); CK(ul(m.box1, S.box1, sl)); CK(ul(m.boxseq, S.boxseq, sl)); CK(ul(m.item0, S.item0, sl)); CK(ul(m.item1, S.item1, sl));
  CK(ul(m.heal, S.heal, sl)); CK(ul(m.healseq, S.healseq, sl)); CK(ul(m.pend0, S.pend0, sl)); CK(ul(m.pend1, S.pend1, sl));
  CK(ul(m.zonec, S.zonec, sl)); CK(ul(m.zonecur, S.zonecur, sl)); CK(ul(m.zoneint, S.zoneint, sl)); CK(ul(m.hdr0, S.hdr0, sl)); CK(ul(m.hdr1, S.hdr1, sl));
  CK(ul(m.pex, S.pex, sl)); CK(ul(m.ptc, S.ptc, sl)); CK(ul(m.pen, S.pen, sl)); CK(ul(m.pseq, S.pseq, sl)); CK(ul(m.pimp, S.pimp, sl));
  CK(ul(m.sreward, S.sreward, sl)); CK(ul(m.skills, S.skills, sl)); CK(ul(m.smisc, S.smisc, sl));
  CK(ul(m.epret, S.epret, sl));
  return MSV_OK;
}
static inline int f2i(float f) { int i; memcpy(&i, &f, 4); return i; }
static inline float i2f(int i) { float f; memcpy(&f, &i, 4); return f; }
static inline bool gbit(const std::vector<unsigned long long>& v, size_t N, size_t e, int p) { return (v[(p >> 6) * N + e] >> (p & 63)) & 1ull; }
static inline void sbit(std::vector<unsigned long long>& v, size_t N, size_t e, int p, bool on) {
  unsigned long long& w = v[(p >> 6) * N + e];
  if (on) w |= 1ull << (p & 63); else w &= ~(1ull << (p & 63));
}


extern "C" {

int msv_abi_version(void) { return MSV_ABI_VERSION; }
int64_t msv_sizeof_config(void) { return (int64_t)sizeof(msv_config); }
int64_t msv_sizeof_env_state(void) { return (int64_t)sizeof(msv_env_state); }
int64_t msv_sizeof_stats(void) { return (int64_t)sizeof(msv_stats); }

int msv_default_config(msv_config* c) {  // env:140-238
  if (!c) return MSV_ERR_INVALID;
  memset(c, 0, sizeof *c);
  c->n_agents = 2; c->n_boxes = 4; c->n_heals = 4; c->teams = 0; c->omniscient = 1;
  c->gameover_mode = MSV_GAMEOVER_ALLDEAD; c->grid_size = 4; c->floor_size = 20;
  c->health = 100; c->melee_range = 2; c->melee_damage = 20; c->melee_cooldown = 40;
  c->box_ownership = 0; c->box_randomized = 0; c->box_health = 20; c->box_size = 1;
  c->box_item_size = 0.5; c->box_item_offset = 0.75; c->heal_item_size = 0.5; c->healing = 50;
  c->inv_slots = 4; c->pickup_radius = 0.5; c->give_radius = 2; c->drop_radius = 0.5;
  c->zone_phases = 5; c->zone_cooldown = 100; c->zone_damage = 1; c->zone_n_radiuses = 4;
  c->zone_radiuses[0] = 10; c->zone_radiuses[1] = 5; c->zone_radiuses[2] = 2.5; c->zone_radiuses[3] = 1;
  c->zone_centers_random = 1;
  c->r_alive = 1; c->r_dead = -1; c->r_kill = 0; c->r_death = 0;
  c->agent_size = 1; c->cam_fov = 0.4 * M_PI; c->cam_depth = 10;
  c->motor_impulse[0] = 0.25; c->motor_impulse[1] = 0.25; c->motor_impulse[2] = 0.0125;
  c->box_min_w = 0.1; c->box_min_h = 0.1;
  c->lidar_n = 0; c->lidar_fov = 0.8 * M_PI; c->lidar_depth = 10;
  c->immunity_cooldown = -1; c->battle_royale = 0; c->b2_variant = 0;
  return MSV_OK;
}

int msv_create(const msv_config* cfg, int32_t num_envs, int32_t device, uint64_t seed, int64_t env_offset,
               msv_handle** out) {
  if (!cfg || !out || num_envs <= 0) return MSV_ERR_INVALID;
  if (cfg->n_agents < 1 || cfg->n_agents > MSV_MAX_AGENTS || cfg->n_boxes < 0 || cfg->n_boxes > MSV_MAX_BOXES ||
      cfg->n_heals < 0 || cfg->n_heals > MSV_MAX_HEALS || cfg->grid_size < 1 || cfg->grid_size > 8 ||
      cfg->n_agents + cfg->n_boxes + cfg->n_heals > cfg->grid_size * cfg->grid_size ||
      cfg->inv_slots < 1 || cfg->inv_slots > MSV_MAX_SLOTS || cfg->zone_n_radiuses + 1 > MSV_MAX_ZONES ||
      cfg->zone_phases > cfg->zone_n_radiuses + 1 || cfg->lidar_n < 0 || cfg->lidar_n > MSV_MAX_LASERS ||
      cfg->zone_phases < 1 || cfg->max_episode_steps < 0 || env_offset < 0 || env_offset + (int64_t)num_envs > (int64_t)1 << 32)   // Philox counter word 0 is 32 bits
    return MSV_ERR_INVALID;
  {  // b2PolygonShape::Set welds vertices closer than its tolerance: a box that small is not a box any more (Box2D asserts);
     // the kernel treats every box analytically, so such configs are refused instead of simulated differently
    const double tol2 = (cfg->b2_variant & MSV_B2_WELD_SQUARED) ? (0.5 * 0.005) * (0.5 * 0.005) : 0.5 * 0.005;   // compared with a SQUARED distance
    const double wmin = cfg->box_randomized ? (cfg->box_min_w < cfg->box_min_h ? cfg->box_min_w : cfg->box_min_h) : cfg->box_size;
    if (cfg->n_boxes > 0 && !(wmin * wmin >= tol2)) { g_err = "box edge below the b2PolygonShape::Set weld tolerance"; return MSV_ERR_INVALID; }
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device >= ndev) {
    g_err = "no CUDA device: libmasurv has no CPU fallback";
    return MSV_ERR_NO_DEVICE;
  }
  msv_handle* h = new msv_handle();
  h->cfg = *cfg; h->device = device; h->launches = 0; h->exported = 0;
  DevGuard guard(device);
  { int cur = -1; if (cudaGetDevice(&cur) != cudaSuccess || cur != device) { delete h; return MSV_ERR_CUDA; } }
  build_const(cfg, num_envs, seed, env_offset, &h->C);
  h->cap = capacity_class(cfg);
  msv_capacity(h->cap, &h->AC, &h->BC, &h->HC, &h->P, &h->PW, &h->sm_words);
  plan_blocks(h, device);
  if (const char* nh = getenv("MSV_NO_HANDOFF")) h->handoff = atoi(nh) == 0;   // development A/B: plain stream-ordered launches
  if (msv_launch(h->cap, 3, h->C, h->S, h->O, nullptr, 0) != cudaSuccess) {
    g_err = "cudaFuncSetAttribute(MaxDynamicSharedMemorySize) failed"; delete h; return MSV_ERR_CUDA;
  }
  const size_t N = (size_t)h->C.N, AC = h->AC, BC = h->BC, HC = h->HC, P = h->P, PW = h->PW;  // padded
  DevState& S = h->S; DevOut& O = h->O;
  int rc = 0;
  rc |= dalloc(h, &S.akin0, AC * N); rc |= dalloc(h, &S.akin1, AC * N); rc |= dalloc(h, &S.afat, AC * N);
  rc |= dalloc(h, &S.aint, AC * N); rc |= dalloc(h, &S.ainv, AC * 4 * N);
  rc |= dalloc(h, &S.box0, BC * N); rc |= dalloc(h, &S.box1, BC * N); rc |= dalloc(h, &S.boxseq, BC * N);
  rc |= dalloc(h, &S.item0, BC * N); rc |= dalloc(h, &S.item1, BC * N);
  rc |= dalloc(h, &S.heal, HC * N); rc |= dalloc(h, &S.healseq, HC * N);
  rc |= dalloc(h, &S.pend0, BC * N); rc |= dalloc(h, &S.pend1, BC * N);
  rc |= dalloc(h, &S.zonec, (size_t)MSV_MAX_ZONES * N); rc |= dalloc(h, &S.zonecur, N); rc |= dalloc(h, &S.zoneint, N);
  rc |= dalloc(h, &S.hdr0, N); rc |= dalloc(h, &S.hdr1, N);
  rc |= dalloc(h, &S.pex, PW * N); rc |= dalloc(h, &S.ptc, PW * N); rc |= dalloc(h, &S.pen, PW * N);
  rc |= dalloc(h, &S.pseq, P * N); rc |= dalloc(h, &S.pimp, P * N);
  rc |= dalloc(h, &S.sreward, AC * N); rc |= dalloc(h, &S.skills, AC * N); rc |= dalloc(h, &S.smisc, N);
  const size_t A = cfg->n_agents, B = cfg->n_boxes, H = cfg->n_heals, Sw = h->C.S, L = cfg->lidar_n;
  rc |= dalloc(h, &S.epret, AC * N);
  rc |= dalloc(h, &S.spare, N * (size_t)MSV_SPARE_W); rc |= dalloc(h, &S.spare_ep, N);
  {  // one arena for every output tensor, so that msv_step_host_obs reads the observations back in ONE copy
    struct Slot { void** p; size_t bytes; };
    const size_t f = sizeof(float);
    Slot slots[] = {
      {(void**)&O.rewards, N * A * f}, {(void**)&O.dones, N}, {(void**)&O.episode_return, N * A * f},
      {(void**)&O.episode_length, N * sizeof(int)}, {(void**)&O.immune, N}, {(void**)&O.br_over, N}, {(void**)&O.br_results, N * A},
      // ---- observation block (obs_begin .. obs_end)
      {(void**)&O.agent, N * A * Sw * f}, {(void**)&O.others, N * A * (A - 1) * Sw * f}, {(void**)&O.others_mask, N * A * (A - 1) * f},
      {(void**)&O.zone, N * 6 * f}, {(void**)&O.heals, N * H * 2 * f}, {(void**)&O.heals_mask, N * A * H * f},
      {(void**)&O.heal_slot, N * A * f}, {(void**)&O.heal_slot_mask, N * A * f}, {(void**)&O.boxes, N * B * 11 * f},
      {(void**)&O.boxes_mask, N * A * B * f}, {(void**)&O.box_items, N * B * 10 * f}, {(void**)&O.box_items_mask, N * A * B * f},
      {(void**)&O.box_slot, N * A * 8 * f}, {(void**)&O.box_slot_mask, N * A * f},
      {(void**)&O.lidar_frac, N * A * L * f}, {(void**)&O.lidar_hit, N * A * L * sizeof(int)},
    };
    const int n_slots = (int)(sizeof slots / sizeof slots[0]), first_obs = 7;
    size_t off = 0; std::vector<size_t> offs;
    for (int k = 0; k < n_slots; ++k) {
      if (k == first_obs) h->obs_begin = off;
      offs.push_back(off);
      off += (slots[k].bytes + 255) / 256 * 256;
    }
    h->obs_end = off; h->arena_bytes = off;
    rc |= dalloc(h, &h->arena, off);
    if (!rc) for (int k = 0; k < n_slots; ++k) *slots[k].p = h->arena + offs[k];
  }
  rc |= dalloc(h, &S.obm, N); rc |= dalloc(h, &S.omask, AC * N);
  rc |= dalloc(h, &S.tq, N / (size_t)h->C.epb); rc |= dalloc(h, &S.tq_tail, 4);
  rc |= dalloc(h, &h->d_actions, N * A * 6);
  if (cfg->max_episode_steps > 0) { rc |= dalloc(h, &h->truncated, N); rc |= dalloc(h, &h->finished, N); }
  rc |= dalloc(h, &h->d_stat_reward, (size_t)MSV_MAX_AGENTS); rc |= dalloc(h, &h->d_stat_kills, (size_t)MSV_MAX_AGENTS);
  rc |= dalloc(h, &h->d_stat_misc, (size_t)4);
  if (rc) { g_err = h->err; msv_destroy(h); return MSV_ERR_ALLOC; }
  {  // episode counter starts at -1 so that the first reset is episode 0
    std::vector<int4> hd(N, make_int4(0, 0, -1, 0));
    cudaMemcpy(S.hdr0, hd.data(), N * sizeof(int4), cudaMemcpyHostToDevice);
    std::vector<int> se(N, INT32_MIN);              // no reset record drawn yet
    cudaMemcpy(S.spare_ep, se.data(), N * sizeof(int), cudaMemcpyHostToDevice);
  }
  {  // the observation keys of k_obs2 (env:391-447 shapes)
    const int Ai = (int)A, Bi = (int)B, Hi = (int)H, Si = (int)Sw;
    ObsKey* K = h->obs.keys;
    K[0] = {O.agent, Ai * Si}; K[1] = {O.others, Ai * (Ai - 1) * Si}; K[2] = {O.others_mask, Ai * (Ai - 1)}; K[3] = {O.zone, 6};
    K[4] = {O.heals, Hi * 2}; K[5] = {O.heals_mask, Ai * Hi}; K[6] = {O.heal_slot, Ai}; K[7] = {O.heal_slot_mask, Ai};
    K[8] = {O.boxes, Bi * 11}; K[9] = {O.boxes_mask, Ai * Bi}; K[10] = {O.box_items, Bi * 10}; K[11] = {O.box_items_mask, Ai * Bi};
    K[12] = {O.box_slot, Ai * 8}; K[13] = {O.box_slot_mask, Ai};
    for (int k = 0; k < MSV_OBS_KEYS; ++k) if (obs_key_used(k, Hi, Bi)) h->obs_floats += K[k].chunk;
    h->obs_term = h->obs;
    if (cfg->auto_reset == 2) {
      for (int k = 0; k < MSV_OBS_KEYS; ++k) {
        float* buf = nullptr;
        if (dalloc(h, &buf, N * (size_t)(K[k].chunk > 0 ? K[k].chunk : 1))) { g_err = h->err; msv_destroy(h); return MSV_ERR_ALLOC; }
        h->obs_term.keys[k].base = buf;
      }
    }
    h->O_term = O;
    if (cfg->auto_reset == 2 && L > 0) {   // the finished episode's last scan, written by a second k_lidar
      if (dalloc(h, &h->O_term.lidar_frac, N * A * L) || dalloc(h, &h->O_term.lidar_hit, N * A * L)) {
        g_err = h->err; msv_destroy(h); return MSV_ERR_ALLOC;
      }
    }
  }
  const int64_t n = num_envs, a = A, b = B, hh = H, s = Sw, l = L;
  reg(h, "agent", O.agent, 0, {n, a, s});
  reg(h, "others", O.others, 0, {n, a, a - 1, s});
  reg(h, "others_mask", O.others_mask, 0, {n, a, a - 1});
  reg(h, "zone", O.zone, 0, {n, 6});
  if (H > 0) {
    reg(h, "heals", O.heals, 0, {n, hh, 2}); reg(h, "heals_mask", O.heals_mask, 0, {n, a, hh});
    reg(h, "heal_slot", O.heal_slot, 0, {n, a, 1, 1}); reg(h, "heal_slot_mask", O.heal_slot_mask, 0, {n, a, 1});
  }
  if (B > 0) {
    reg(h, "boxes", O.boxes, 0, {n, b, 11}); reg(h, "boxes_mask", O.boxes_mask, 0, {n, a, b});
    reg(h, "box_items", O.box_items, 0, {n, b, 10}); reg(h, "box_items_mask", O.box_items_mask, 0, {n, a, b});
    reg(h, "box_slot", O.box_slot, 0, {n, a, 1, 8}); reg(h, "box_slot_mask", O.box_slot_mask, 0, {n, a, 1});
  }
  if (L > 0) { reg(h, "lidar_frac", O.lidar_frac, 0, {n, a, l}); reg(h, "lidar_hit", O.lidar_hit, 2, {n, a, l}); }
  reg(h, "rewards", O.rewards, 0, {n, a});
  reg(h, "dones", O.dones, 1, {n});
  reg(h, "episode_return", O.episode_return, 0, {n, a});
  reg(h, "episode_length", O.episode_length, 2, {n});
  if (cfg->immunity_cooldown >= 0) reg(h, "immune", O.immune, 1, {n});
  if (cfg->battle_royale) { reg(h, "br_over", O.br_over, 1, {n}); reg(h, "br_results", O.br_results, 1, {n, a}); }
  if (cfg->max_episode_steps > 0) reg(h, "truncated", h->truncated, 1, {n});
  if (cfg->auto_reset == 2) {   // same shapes, "terminal_" prefix
    std::map<std::string, TensorInfo> extra;
    static const char* names[MSV_OBS_KEYS] = {"agent", "others", "others_mask", "zone", "heals", "heals_mask", "heal_slot",
                                              "heal_slot_mask", "boxes", "boxes_mask", "box_items", "box_items_mask", "box_slot", "box_slot_mask"};
    for (int k = 0; k < MSV_OBS_KEYS; ++k) {
      auto it = h->tensors.find(names[k]);
      if (it == h->tensors.end()) continue;
      TensorInfo t = it->second; t.ptr = h->obs_term.keys[k].base;
      extra[std::string("terminal_") + names[k]] = t;
    }
    if (L > 0) {
      extra["terminal_lidar_frac"] = h->tensors["lidar_frac"]; extra["terminal_lidar_frac"].ptr = h->O_term.lidar_frac;
      extra["terminal_lidar_hit"] = h->tensors["lidar_hit"]; extra["terminal_lidar_hit"].ptr = h->O_term.lidar_hit;
    }
    for (auto& kv : extra) h->tensors[kv.first] = kv.second;
  }
  *out = h;
  return MSV_OK;
}

static void really_destroy(msv_handle* h) {
  DevGuard g(h->device);
  cudaDeviceSynchronize();
  for (void* p : h->allocs) cudaFree(p);
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  if (h->side_stream) cudaStreamDestroy(h->side_stream);
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  if (h->ev_step) cudaEventDestroy(h->ev_step);
  if (h->ev_obs) cudaEventDestroy(h->ev_obs);
  if (h->ev_copy) cudaEventDestroy(h->ev_copy);
  if (h->ev_up) cudaEventDestroy(h->ev_up);
  if (h->ev_done) cudaEventDestroy(h->ev_done);
  if (h->up_stream) cudaStreamDestroy(h->up_stream);
  for (cudaEvent_t e : h->tev) cudaEventDestroy(e);
  delete h;
}

int msv_destroy(msv_handle* h) {
  if (!h || h->zombie) return MSV_ERR_INVALID;
  if (h->exported > 0) {          // tensors handed out through DLPack are still alive: their
    DevGuard g(h->device);        // storage (and the handle their deleter refers to) stays until
    cudaDeviceSynchronize();      // the last one is deleted (dl_deleter)
    h->zombie = true;
    return MSV_OK;
  }
  really_destroy(h);
  return MSV_OK;
}

const char* msv_last_error(msv_handle* h) { return h ? h->err.c_str() : g_err.c_str(); }

// ---- host read-back (msv_step_host*) ----------------------------------------
static int copy_setup(msv_handle* h) {
  if (h->copy_stream) return MSV_OK;
  CK(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
  CK(cudaEventCreateWithFlags(&h->ev_step, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&h->ev_obs, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&h->ev_copy, cudaEventDisableTiming));
  CK(cudaStreamCreateWithFlags(&h->up_stream, cudaStreamNonBlocking));
  CK(cudaEventCreateWithFlags(&h->ev_up, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&h->ev_done, cudaEventDisableTiming));
  return MSV_OK;
}
// rewards and dones are final once the step kernel has run: copy them to the host buffers of a
// pending msv_step_host on the copy stream while the observation kernels run on `st`
static int readback(msv_handle* h, cudaStream_t st) {
  if (!h->host_rewards && !h->host_dones) return MSV_OK;
  size_t N = h->C.n_real, A = h->C.A;
  CK(cudaEventRecord(h->ev_step, st));
  CK(cudaStreamWaitEvent(h->copy_stream, h->ev_step, 0));
  if (h->host_rewards) CK(cudaMemcpyAsync(h->host_rewards, h->O.rewards, N * A * sizeof(float), cudaMemcpyDeviceToHost, h->copy_stream));
  if (h->host_dones) CK(cudaMemcpyAsync(h->host_dones, h->O.dones, N, cudaMemcpyDeviceToHost, h->copy_stream));
  return MSV_OK;
}
// the observation arena, once the observation kernels are done
static int readback_obs(msv_handle* h, cudaStream_t st) {
  if (h->host_obs) {
    CK(cudaEventRecord(h->ev_obs, st));
    CK(cudaStreamWaitEvent(h->copy_stream, h->ev_obs, 0));
    CK(cudaMemcpyAsync(h->host_obs, h->arena + h->obs_begin, h->obs_end - h->obs_begin, cudaMemcpyDeviceToHost, h->copy_stream));
  }
  if (h->host_obs || h->host_rewards || h->host_dones) {
    CK(cudaEventRecord(h->ev_copy, h->copy_stream));
    h->copy_pending = true;
  }
  return MSV_OK;
}

// debug kernel timing: one event before and one after every kernel of a step
static void tmark(msv_handle* h, cudaStream_t st) {
  if (!h->timing) return;
  if (h->tev_used >= h->tev.size()) {
    if (h->tev.size() >= 4 * 8192) { h->timing = false; return; }
    cudaEvent_t e; if (cudaEventCreate(&e) != cudaSuccess) { h->timing = false; return; }
    h->tev.push_back(e);
  }
  cudaEventRecord(h->tev[h->tev_used++], st);
}

// which: 0 step (dev_in = the actions), 1 reset (dev_in = the mask of the envs to reset, NULL = every env), 2 observe
static int launch(msv_handle* h, int which, const uint8_t* dev_in, void* stream) {
  DevGuard g(h->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (h->copy_pending) {                        // a read-back of the previous step may still be reading the arena
    h->copy_pending = false;
    CK(cudaStreamWaitEvent(st, h->ev_copy, 0));
  }
  const bool timed = h->timing && which == 0;
  if (timed) tmark(h, st);
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  const bool capturing = cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone;
  // Terminal capture and the step limit split the step: k_step without the in-kernel reset, then the kernels that
  // need the finished episodes' last state, then the reset of the finished environments.
  const int T = h->cfg.max_episode_steps;
  const bool split = which == 0 && (h->cfg.auto_reset == 2 || T > 0);
  // Tile hand-off (DevConst::tq_ticket): the observation kernel is launched programmatically dependent on the
  // step kernel and consumes the step kernel's blocks in the order they finish, so the observation of a finished
  // tile is written while the step's slow blocks (a wedged agent, a multi-agent island, a reset) still run.
  // Needs the two launches adjacent in the stream: off under kernel timing, stream capture and a split step.
  DevConst Cq = h->C;
  const bool handoff = which == 0 && !split && !timed && !capturing && h->handoff;
  if (handoff) {
    if (++h->tq_ticket == 0u) h->tq_ticket = 1u;
    Cq.tq_ticket = h->tq_ticket; Cq.tq_base = h->tq_base;
    Cq.pdl_wait = (h->last_was_step && h->last_stream == st) ? 1u : 0u;   // the previous call on this stream ended with this handle's observation kernels
    h->tq_base += (uint32_t)(h->C.N / h->C.epb);
  }
  if (split) {
    // step without the in-kernel reset; flag the episodes the step limit ends (finished = dones | truncated); keep
    // the finished episodes' last observation; reset exactly the finished envs (same Philox streams as the in-kernel reset)
    DevConst C0 = h->C; C0.auto_reset = 0;
    CK(msv_launch(h->cap, 0, C0, h->S, h->O, dev_in, st));
    h->launches += 1;
    { int rc = readback(h, st); if (rc) return rc; }
    const uint8_t* fin = h->O.dones;
    if (T > 0) {
      CK(msv_launch_truncate(h->C, h->S, h->O, T, h->truncated, h->finished, st));
      h->launches += 1;
      fin = h->finished;
    }
    if (h->cfg.auto_reset == 2) {
      CK(msv_launch_obs(h->C, h->S, h->obs_term, h->AC, fin, st));
      h->launches += 1;
      if (h->C.lidar_n > 0) { CK(msv_launch_lidar(h->C, h->S, h->O_term, h->BC, h->HC, st)); h->launches++; }
    }
    if (h->cfg.auto_reset != 0) {
      CK(msv_launch_reset(h->cap, h->C, h->S, h->O, fin, 1, nullptr, st));
      h->launches += 1;
    }
  } else if (which == 1) {
    // observations are a pure function of the state: the unmasked rows of a masked reset are rewritten with the
    // values they already hold by the full observation pass below
    CK(msv_launch_reset(h->cap, h->C, h->S, h->O, dev_in, 0, h->truncated, st));
    h->launches += 1;
  } else {
    CK(msv_launch(h->cap, which, Cq, h->S, h->O, dev_in, st));
    h->launches += 1;
    if (which == 0 && !handoff) { int rc = readback(h, st); if (rc) return rc; }
  }
  if (timed) tmark(h, st);
  CK(msv_launch_obs(Cq, h->S, h->obs, h->AC, nullptr, st));   // fetch_observations
  h->launches += 1;
  if (which == 0 && handoff) { int rc = readback(h, st); if (rc) return rc; }   // (an event between the two launches would serialise them)
  if (timed) tmark(h, st);
  if (h->C.lidar_n > 0) { CK(msv_launch_lidar(h->C, h->S, h->O, h->BC, h->HC, (cudaStream_t)stream)); h->launches++; }
  if (timed) tmark(h, st);
  const bool spare = which == 1 || (which == 0 && h->cfg.auto_reset != 0);
  if (spare) {                                  // the step / reset left finished environments without a record for their next episode
    if (!h->side_stream) {
      CK(cudaStreamCreateWithFlags(&h->side_stream, cudaStreamNonBlocking));
      CK(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
      CK(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    }
    // The record kernel runs on a side stream, forked after the observation kernels and NOT joined back in normal
    // operation: it overlaps the next step, and nothing on `st` ever waits for it.  That is safe by construction --
    // a record is published by writing its episode number last (after a fence); a reset that does not find the
    // number it expects draws the record itself -- and msv_get_state / msv_set_state / msv_destroy synchronise
    // the device.  Only while the caller is capturing `st` into a CUDA graph must the fork be joined inside the call.
    CK(cudaEventRecord(h->ev_fork, st));
    CK(cudaStreamWaitEvent(h->side_stream, h->ev_fork, 0));
    CK(msv_launch_spare(h->C, h->S, h->O.dones, 0, h->side_stream));   // every env whose record is stale (two 4-byte loads each for the others)
    CK(cudaEventRecord(h->ev_join, h->side_stream));
    h->launches += 1;
    if (capturing) CK(cudaStreamWaitEvent(st, h->ev_join, 0));
  }
  if (which == 0) { int rc = readback_obs(h, st); if (rc) return rc; }
  h->last_was_step = handoff; h->last_stream = st;
  return MSV_OK;
}

/* debug: number of capacity-overflow events (contact list, TOI island, item
 * lists) any env has recorded since its last set_state -- must stay 0 */
int64_t msv_debug_overflow(msv_handle* h) {
  if (!h) return -1;
  DevGuard g(h->device); cudaDeviceSynchronize();
  std::vector<int4> v((size_t)h->C.N);
  if (cudaMemcpy(v.data(), h->S.hdr1, v.size() * sizeof(int4), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  int64_t tot = 0;
  for (int e = 0; e < h->C.n_real; ++e) tot += v[e].z;
  unsigned tq[4] = {0, 0, 0, 0};                  // [2]: an observation tile gave up waiting for its completion-queue entry
  if (cudaMemcpy(tq, h->S.tq_tail, sizeof tq, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  if (tq[2]) tot += 1000000;
  return tot;
}

/* debug: bounds-check violations counted by a `make CHECK=1` build since the library was loaded
 * (-1: error, -2: this is not a checked build); *line = source line of the last violation */
int64_t msv_debug_check_failures(msv_handle* h, int64_t* line) {
  if (!h) return -1;
  DevGuard g(h->device); cudaDeviceSynchronize();
  unsigned long long v[2] = {0, 0};
  if (msv_read_check(v) != cudaSuccess) return -1;
  if (line) *line = (int64_t)v[1];
  return v[0] == ~0ull ? -2 : (int64_t)v[0];
}

/* debug/bench: the two halves of msv_step separately, so that bench.py can put
 * CUDA events around the dominant kernel alone */
int msv_debug_step_kernel(msv_handle* h, const uint8_t* actions_dev, void* stream) {
  if (!h || !actions_dev) return MSV_ERR_INVALID;
  CK(msv_launch(h->cap, 0, h->C, h->S, h->O, actions_dev, (cudaStream_t)stream));
  h->launches++;
  return MSV_OK;
}
int msv_debug_obs_kernel(msv_handle* h, void* stream) {
  if (!h) return MSV_ERR_INVALID;
  CK(msv_launch_obs(h->C, h->S, h->obs, h->AC, nullptr, (cudaStream_t)stream));
  h->launches++;
  return MSV_OK;
}

int msv_reset(msv_handle* h, void* stream) { return h ? launch(h, 1, nullptr, stream) : MSV_ERR_INVALID; }
int msv_reset_envs(msv_handle* h, const uint8_t* mask_dev, void* stream) {
  if (!h || !mask_dev) return MSV_ERR_INVALID;
  return launch(h, 1, mask_dev, stream);
}
int msv_observe(msv_handle* h, void* stream) { return h ? launch(h, 2, nullptr, stream) : MSV_ERR_INVALID; }
int msv_step(msv_handle* h, const uint8_t* actions_dev, void* stream) {
  if (!h || !actions_dev) return MSV_ERR_INVALID;
  return launch(h, 0, actions_dev, stream);
}

int msv_render(msv_handle* h, int32_t first, int32_t count, int32_t height, int32_t width, uint32_t flags,
               uint8_t* out_dev, void* stream) {
  if (!h || !out_dev) return MSV_ERR_INVALID;
  if (first < 0 || count < 1 || (int64_t)first + count > h->C.n_real || height < 1 || height > 4096 || width < 1 ||
      width > 4096 || (flags & ~MSV_RENDER_LIDAR) || ((flags & MSV_RENDER_LIDAR) && h->C.lidar_n == 0)) {
    h->err = "msv_render: env range, image size (1..4096) or flags out of range";
    return MSV_ERR_INVALID;
  }
  DevGuard g(h->device);
  RenderArgs R = {};
  R.first = first; R.count = count; R.H = height; R.W = width; R.BC = h->BC; R.HC = h->HC;
  R.lidar = (flags & MSV_RENDER_LIDAR) ? 1 : 0; R.out = out_dev;
  const cudaError_t e = msv_launch_render(h->C, h->S, h->O, R, (cudaStream_t)stream);
  h->launches++;
  h->last_was_step = false;    // the next k_step must not wait for an observation kernel that is not the last launch
  CK(e);
  return MSV_OK;
}

int msv_render_palette(uint8_t* out_rgb, int32_t capacity) {
  if (capacity < 0 || (capacity > 0 && !out_rgb)) return MSV_ERR_INVALID;
  return msv_palette(out_rgb, capacity);
}

int msv_step_host_async(msv_handle* h, const uint8_t* actions_host, float* rewards_host, uint8_t* dones_host, void* obs_host,
                        void* stream) {
  if (!h || !actions_host) return MSV_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  size_t N = h->C.n_real, A = h->C.A;
  DevGuard g(h->device);
  { int rc = copy_setup(h); if (rc) return rc; }
  if (h->copy_pending) {       // d_actions / the arena are reused: order this step after the previous read-back
    h->copy_pending = false;
    CK(cudaStreamWaitEvent(st, h->ev_copy, 0));
  }
  // upload on up_stream: after this handle's previous step (whose step kernel read d_actions), before this one's
  if (h->done_valid) CK(cudaStreamWaitEvent(h->up_stream, h->ev_done, 0));
  cudaError_t ce = cudaMemcpyAsync(h->d_actions, actions_host, N * A * 6, cudaMemcpyHostToDevice, h->up_stream);
  int rc = MSV_OK;
  if (ce != cudaSuccess) { h->err = std::string("cudaMemcpyAsync(actions): ") + cudaGetErrorString(ce); rc = MSV_ERR_CUDA; }
  if (!rc && (cudaEventRecord(h->ev_up, h->up_stream) != cudaSuccess || cudaStreamWaitEvent(st, h->ev_up, 0) != cudaSuccess)) {
    h->err = "cudaEventRecord/cudaStreamWaitEvent(upload) failed"; rc = MSV_ERR_CUDA;
  }
  if (!rc) {
    h->host_rewards = rewards_host; h->host_dones = dones_host; h->host_obs = obs_host;
    rc = launch(h, 0, h->d_actions, stream);
    h->host_rewards = nullptr; h->host_dones = nullptr; h->host_obs = nullptr;
  }
  if (!rc) { if (cudaEventRecord(h->ev_done, st) == cudaSuccess) h->done_valid = true; else { h->err = "cudaEventRecord(step done) failed"; rc = MSV_ERR_CUDA; } }
  if (rc) {                    // nothing may still be writing into the caller's buffers after an error return
    cudaStreamSynchronize(h->up_stream); cudaStreamSynchronize(h->copy_stream); cudaStreamSynchronize(st);
    h->copy_pending = false;
  }
  return rc;
}

int msv_step_host_wait(msv_handle* h) {
  if (!h) return MSV_ERR_INVALID;
  if (!h->copy_stream || !h->copy_pending) return MSV_OK;
  DevGuard g(h->device);
  // spin on the copy-out event: no blocking stream synchronize on the launch stream
  for (;;) {
    cudaError_t e = cudaEventQuery(h->ev_copy);
    if (e == cudaSuccess) break;
    if (e != cudaErrorNotReady) { h->err = std::string("cudaEventQuery: ") + cudaGetErrorString(e); h->copy_pending = false; return MSV_ERR_CUDA; }
  }
  // copy_pending stays set: the next launch on the handle makes its stream wait for the (completed) event
  return MSV_OK;
}

int msv_step_host(msv_handle* h, const uint8_t* actions_host, float* rewards_host, uint8_t* dones_host, void* stream) {
  int rc = msv_step_host_async(h, actions_host, rewards_host, dones_host, nullptr, stream);
  if (rc) return rc;
  rc = msv_step_host_wait(h);
  if (rc) return rc;
  DevGuard g(h->device);
  CK(cudaStreamSynchronize((cudaStream_t)stream));   // observation tensors complete as well (documented contract)
  return MSV_OK;
}

int msv_step_host_obs(msv_handle* h, const uint8_t* actions_host, float* rewards_host, uint8_t* dones_host, void* obs_host,
                      void* stream) {
  if (!obs_host) return MSV_ERR_INVALID;
  int rc = msv_step_host_async(h, actions_host, rewards_host, dones_host, obs_host, stream);
  if (rc) return rc;
  return msv_step_host_wait(h);
}

int64_t msv_obs_host_bytes(msv_handle* h) { return h ? (int64_t)(h->obs_end - h->obs_begin) : 0; }
int64_t msv_obs_host_offset(msv_handle* h, const char* name) {
  if (!h || !name) return -1;
  auto it = h->tensors.find(name);
  if (it == h->tensors.end()) return -1;
  const char* p = (const char*)it->second.ptr;
  if (p < h->arena + h->obs_begin || p >= h->arena + h->obs_end) return -1;
  return (int64_t)(p - (h->arena + h->obs_begin));
}
int64_t msv_device_bytes(msv_handle* h) { return h ? (int64_t)h->device_bytes : 0; }

/* debug/bench: CUDA-event timing of the kernels msv_step launches.  enable=1 starts recording (one
 * event pair per kernel and step, up to 8192 steps); enable=0 stops, synchronises and returns the
 * mean milliseconds of [k_step (+ terminal capture), k_obs2, k_lidar] and the number of steps. */
int msv_debug_kernel_timing(msv_handle* h, int enable, double out_ms[3], int64_t* n_steps) {
  if (!h) return MSV_ERR_INVALID;
  DevGuard g(h->device);
  if (enable) { h->tev_used = 0; h->timing = true; return MSV_OK; }
  h->timing = false;
  CK(cudaDeviceSynchronize());
  double sum[3] = {0, 0, 0}; int64_t n = (int64_t)(h->tev_used / 4);
  for (int64_t t = 0; t < n; ++t)
    for (int k = 0; k < 3; ++k) {
      float ms = 0.0f; CK(cudaEventElapsedTime(&ms, h->tev[4 * t + k], h->tev[4 * t + k + 1]));
      sum[k] += ms;
    }
  if (out_ms) for (int k = 0; k < 3; ++k) out_ms[k] = n ? sum[k] / (double)n : 0.0;
  if (n_steps) *n_steps = n;
  h->tev_used = 0;
  return MSV_OK;
}

int msv_tensor_info(msv_handle* h, const char* name, void** dev_ptr, int32_t* ndim, int64_t shape[4],
                    int64_t strides[4], int32_t* dtype_code) {
  if (!h || !name) return MSV_ERR_INVALID;
  auto it = h->tensors.find(name);
  if (it == h->tensors.end()) { h->err = std::string("unknown tensor: ") + name; return MSV_ERR_NAME; }
  const TensorInfo& t = it->second;
  if (dev_ptr) *dev_ptr = t.ptr;
  if (ndim) *ndim = t.ndim;
  int64_t st = 1;
  for (int i = t.ndim - 1; i >= 0; --i) { if (shape) shape[i] = t.shape[i]; if (strides) strides[i] = st; st *= t.shape[i]; }
  if (dtype_code) *dtype_code = t.dtype;
  return MSV_OK;
}

struct DLCtx { msv_handle* h; int64_t shape[4]; int64_t strides[4]; };
static void dl_deleter(DLManagedTensor* m) {
  if (!m) return;
  DLCtx* c = (DLCtx*)m->manager_ctx;
  // the library owns the memory for the handle's lifetime: only drop the count
  if (c) {
    msv_handle* h = c->h;
    delete c;
    if (--h->exported == 0 && h->zombie) really_destroy(h);
  }
  delete m;
}

int msv_tensor(msv_handle* h, const char* name, struct DLManagedTensor** out) {
  if (!h || !name || !out) return MSV_ERR_INVALID;
  auto it = h->tensors.find(name);
  if (it == h->tensors.end()) { h->err = std::string("unknown tensor: ") + name; return MSV_ERR_NAME; }
  const TensorInfo& t = it->second;
  DLCtx* c = new DLCtx(); c->h = h;
  int64_t st = 1;
  for (int i = t.ndim - 1; i >= 0; --i) { c->shape[i] = t.shape[i]; c->strides[i] = st; st *= t.shape[i]; }
  DLManagedTensor* m = new DLManagedTensor();
  m->dl_tensor.data = t.ptr;
  m->dl_tensor.device.device_type = 2;  // kDLCUDA
  m->dl_tensor.device.device_id = h->device;
  m->dl_tensor.ndim = t.ndim;
  m->dl_tensor.dtype.code = t.dtype == 0 ? 2 : (t.dtype == 1 ? 1 : 0);  // kDLFloat / kDLUInt / kDLInt
  m->dl_tensor.dtype.bits = t.dtype == 1 ? 8 : 32;
  m->dl_tensor.dtype.lanes = 1;
  m->dl_tensor.shape = c->shape; m->dl_tensor.strides = c->strides; m->dl_tensor.byte_offset = 0;
  m->manager_ctx = c; m->deleter = dl_deleter;
  h->exported++;
  *out = m;
  return MSV_OK;
}

int msv_get_state(msv_handle* h, int32_t first, int32_t count, msv_env_state* out) {
  if (!h || !out || first < 0 || count < 0 || first + count > h->C.n_real) return MSV_ERR_INVALID;
  if (count == 0) return MSV_OK;
  DevGuard g(h->device);
  const Slice sl{(size_t)first, (size_t)count, (size_t)h->C.N};
  Mirror m; int rc = download(h, m, sl); if (rc) return rc;
  const size_t N = (size_t)count; const int AC = h->AC, BC = h->BC, A = h->C.A, NAA = AC * (AC - 1) / 2;
  for (int q = 0; q < count; ++q) {
    size_t e = (size_t)q; msv_env_state& s = out[q];
    memset(&s, 0, sizeof s);
    for (int i = 0; i < A; ++i) {
      float4 k0 = m.akin0[i * N + e], k1 = m.akin1[i * N + e], ft = m.afat[i * N + e]; int4 ai = m.aint[i * N + e];
      int fl = f2i(k1.w);
      s.alive[i] = fl & 1; s.cooldown[i] = ai.z; s.cause[i] = MSV_CAUSE_NONE;
      if (!s.alive[i]) continue;
      s.awake[i] = (fl >> 1) & 1;
      s.x[i] = k0.x; s.y[i] = k0.y; s.angle[i] = k0.z; s.vx[i] = k0.w; s.vy[i] = k1.x; s.omega[i] = k1.y; s.sleep_time[i] = k1.z;
      s.fat[i][0] = ft.x; s.fat[i][1] = ft.y; s.fat[i][2] = ft.z; s.fat[i][3] = ft.w;
      s.health[i] = ai.x; s.cause[i] = ai.y;
      s.inv_n[i] = ai.w & 7;
      for (int k = 0; k < s.inv_n[i]; ++k) {
        s.inv_kind[i][k] = (ai.w >> (4 + 2 * k)) & 3;
        s.inv_owner[i][k] = MSV_CAUSE_NONE;
        if (s.inv_kind[i][k] == MSV_ITEM_BOX) {
          float4 pl = m.ainv[(i * 4 + k) * N + e];
          s.inv_shape[i][k].hx = pl.x; s.inv_shape[i][k].hy = pl.y; s.inv_owner[i][k] = f2i(pl.z); s.inv_shape[i][k].rehulled = f2i(pl.w) & 1;
        }
      }
    }
    int4 h0 = m.hdr0[e], h1 = m.hdr1[e];
    s.n_boxes = h0.x & 255; s.n_items = (h0.x >> 8) & 255; s.n_heals = (h0.x >> 16) & 255; s.n_pending = (h0.x >> 24) & 255;
    for (int k = 0; k < s.n_boxes; ++k) {
      float4 b0 = m.box0[k * N + e]; int4 b1 = m.box1[k * N + e];
      s.box_x[k] = b0.x; s.box_y[k] = b0.y; s.box_shape[k].hx = b0.z; s.box_shape[k].hy = b0.w; s.box_shape[k].rehulled = (b1.y >> 1) & 1;
      s.box_health[k] = b1.x; s.box_has_health[k] = b1.y & 1; s.box_cause[k] = b1.z; s.box_owner[k] = b1.w; s.box_seq[k] = m.boxseq[k * N + e];
    }
    for (int k = 0; k < s.n_items; ++k) {
      float4 i0 = m.item0[k * N + e]; int2 i1 = m.item1[k * N + e];
      s.item_x[k] = i0.x; s.item_y[k] = i0.y; s.item_shape[k].hx = i0.z; s.item_shape[k].hy = i0.w; s.item_shape[k].rehulled = 1;
      s.item_owner[k] = i1.x; s.item_seq[k] = i1.y;
    }
    for (int k = 0; k < s.n_heals; ++k) { float2 hh = m.heal[k * N + e]; s.heal_x[k] = hh.x; s.heal_y[k] = hh.y; s.heal_seq[k] = m.healseq[k * N + e]; }
    for (int k = 0; k < s.n_pending; ++k) {
      float4 p0 = m.pend0[k * N + e];
      s.pend_x[k] = p0.x; s.pend_y[k] = p0.y; s.pend_shape[k].hx = p0.z; s.pend_shape[k].hy = p0.w; s.pend_shape[k].rehulled = 1;
      s.pend_owner[k] = m.pend1[k * N + e];
    }
    for (int z = 0; z < h->C.n_zones; ++z) { float2 zc = m.zonec[z * N + e]; s.zone_cx[z] = zc.x; s.zone_cy[z] = zc.y; }
    int4 zi = m.zoneint[e]; float4 zc = m.zonecur[e];
    s.zone_phase = zi.x; s.zone_t_cooldown = zi.y; s.zone_t_shrink = zi.z; s.zone_endgame = zi.w;
    s.zone_cur_x = zc.x; s.zone_cur_y = zc.y; s.zone_cur_r = zc.z;
    auto get_pair = [&](int p, msv_pair& pr) {
      if (!gbit(m.pex, N, e, p)) return;
      pr.seq = (int32_t)m.pseq[p * N + e];
      pr.flags = (gbit(m.ptc, N, e, p) ? MSV_PAIR_TOUCHING : 0) | (gbit(m.pen, N, e, p) ? MSV_PAIR_ENABLED : 0);
      float2 im = m.pimp[p * N + e]; pr.normal_impulse = im.x; pr.tangent_impulse = im.y;
    };
    for (int j = 1; j < A; ++j) for (int i = 0; i < j; ++i) get_pair(j * (j - 1) / 2 + i, s.pair_aa[j * (j - 1) / 2 + i]);
    for (int i = 0; i < A; ++i) {
      for (int k = 0; k < s.n_boxes; ++k) get_pair(NAA + i * BC + k, s.pair_ab[i][k]);
      for (int k = 0; k < 4; ++k) get_pair(NAA + AC * BC + i * 4 + k, s.pair_aw[i][k]);
    }
    s.first_step = h1.y; s.steps = h0.y; s.episode = h0.z; s.body_seq = h0.w; s.contact_seq = h1.x;
    for (int i = 0; i < AC; ++i) { s.stat_reward[i] = m.sreward[i * N + e]; s.stat_kills[i] = m.skills[i * N + e]; }
    int4 sm = m.smisc[e]; s.stat_steps = sm.x; s.stat_heals_used = sm.y; s.stat_boxes_placed = sm.z; s.stat_episodes = sm.w;
    for (int i = 0; i < A; ++i) s.ep_return[i] = m.epret[i * N + e];
  }
  return MSV_OK;
}

int msv_set_state(msv_handle* h, int32_t first, int32_t count, const msv_env_state* in) {
  if (!h || !in || first < 0 || count < 0 || first + count > h->C.n_real) return MSV_ERR_INVALID;
  if (count == 0) return MSV_OK;
  const int AC = h->AC, BC = h->BC, HC = h->HC, A = h->C.A, NAA = AC * (AC - 1) / 2;
  for (int q = 0; q < count; ++q) {   // validate everything before touching the device
    const msv_env_state& s = in[q];
    bool ok = s.n_boxes >= 0 && s.n_boxes <= BC && s.n_items >= 0 && s.n_items <= BC && s.n_heals >= 0 && s.n_heals <= HC &&
              s.n_pending >= 0 && s.n_pending <= BC && s.zone_phase >= 0 && s.zone_phase < h->C.zone_phases &&
              s.n_boxes + s.n_pending <= 255;
    for (int i = 0; ok && i < A; ++i) {
      ok = s.inv_n[i] >= 0 && s.inv_n[i] <= h->C.inv_slots;
      for (int k = 0; ok && k < s.inv_n[i]; ++k) ok = s.inv_kind[i][k] == MSV_ITEM_HEAL || s.inv_kind[i][k] == MSV_ITEM_BOX;
    }
    if (!ok) { h->err = "msv_set_state: list length / inventory / zone phase out of range in env record " + std::to_string(q); return MSV_ERR_INVALID; }
  }
  DevGuard g(h->device);
  const Slice sl{(size_t)first, (size_t)count, (size_t)h->C.N};
  Mirror m; int rc = download(h, m, sl); if (rc) return rc;
  const size_t N = (size_t)count;
  for (int q = 0; q < count; ++q) {
    size_t e = (size_t)q; const msv_env_state& s = in[q];
    for (int i = 0; i < A; ++i) {
      int fl = (s.alive[i] ? 1 : 0) | (s.alive[i] && s.awake[i] ? 2 : 0);
      m.akin0[i * N + e] = make_float4(s.x[i], s.y[i], s.angle[i], s.vx[i]);
      m.akin1[i * N + e] = make_float4(s.vy[i], s.omega[i], s.sleep_time[i], i2f(fl));
      m.afat[i * N + e] = make_float4(s.fat[i][0], s.fat[i][1], s.fat[i][2], s.fat[i][3]);
      int inv = s.alive[i] ? s.inv_n[i] : 0;
      for (int k = 0; k < (s.alive[i] ? s.inv_n[i] : 0); ++k) {
        inv |= s.inv_kind[i][k] << (4 + 2 * k);
        m.ainv[(i * 4 + k) * N + e] = make_float4(s.inv_shape[i][k].hx, s.inv_shape[i][k].hy, i2f(s.inv_owner[i][k]), i2f(s.inv_shape[i][k].rehulled));
      }
      m.aint[i * N + e] = make_int4(s.health[i], s.cause[i], s.cooldown[i], inv);
    }
    m.hdr0[e] = make_int4(s.n_boxes | (s.n_items << 8) | (s.n_heals << 16) | (s.n_pending << 24), s.steps, s.episode, s.body_seq);
    m.hdr1[e] = make_int4(s.contact_seq, s.first_step, 0, 1);   // .w: new fixtures -> the next Step searches for contacts first
    for (int k = 0; k < s.n_boxes; ++k) {
      m.box0[k * N + e] = make_float4(s.box_x[k], s.box_y[k], s.box_shape[k].hx, s.box_shape[k].hy);
      m.box1[k * N + e] = make_int4(s.box_health[k], (s.box_has_health[k] ? 1 : 0) | (s.box_shape[k].rehulled ? 2 : 0), s.box_cause[k], s.box_owner[k]);
      m.boxseq[k * N + e] = s.box_seq[k];
    }
    for (int k = 0; k < s.n_items; ++k) {
      m.item0[k * N + e] = make_float4(s.item_x[k], s.item_y[k], s.item_shape[k].hx, s.item_shape[k].hy);
      m.item1[k * N + e] = make_int2(s.item_owner[k], s.item_seq[k]);
    }
    for (int k = 0; k < s.n_heals; ++k) { m.heal[k * N + e] = make_float2(s.heal_x[k], s.heal_y[k]); m.healseq[k * N + e] = s.heal_seq[k]; }
    for (int k = 0; k < s.n_pending; ++k) {
      m.pend0[k * N + e] = make_float4(s.pend_x[k], s.pend_y[k], s.pend_shape[k].hx, s.pend_shape[k].hy);
      m.pend1[k * N + e] = s.pend_owner[k];
    }
    for (int z = 0; z < h->C.n_zones; ++z) m.zonec[z * N + e] = make_float2(s.zone_cx[z], s.zone_cy[z]);
    m.zoneint[e] = make_int4(s.zone_phase, s.zone_t_cooldown, s.zone_t_shrink, s.zone_endgame);
    m.zonecur[e] = make_float4(s.zone_cur_x, s.zone_cur_y, s.zone_cur_r, 0.0f);
    for (int p = 0; p < h->P; ++p) { sbit(m.pex, N, e, p, false); sbit(m.ptc, N, e, p, false); sbit(m.pen, N, e, p, false); }
    auto set_pair = [&](int p, const msv_pair& pr) {
      if (!pr.seq) return;
      sbit(m.pex, N, e, p, true); sbit(m.ptc, N, e, p, pr.flags & MSV_PAIR_TOUCHING); sbit(m.pen, N, e, p, pr.flags & MSV_PAIR_ENABLED);
      m.pseq[p * N + e] = (uint32_t)pr.seq; m.pimp[p * N + e] = make_float2(pr.normal_impulse, pr.tangent_impulse);
    };
    for (int j = 1; j < A; ++j) for (int i = 0; i < j; ++i)
      if (s.alive[i] && s.alive[j]) set_pair(j * (j - 1) / 2 + i, s.pair_aa[j * (j - 1) / 2 + i]);
    for (int i = 0; i < A; ++i) {
      if (!s.alive[i]) continue;
      for (int k = 0; k < s.n_boxes; ++k) set_pair(NAA + i * BC + k, s.pair_ab[i][k]);
      for (int k = 0; k < 4; ++k) set_pair(NAA + AC * BC + i * 4 + k, s.pair_aw[i][k]);
    }
    for (int i = 0; i < AC; ++i) { m.sreward[i * N + e] = s.stat_reward[i]; m.skills[i * N + e] = s.stat_kills[i]; }
    m.smisc[e] = make_int4(s.stat_steps, s.stat_heals_used, s.stat_boxes_placed, s.stat_episodes);
    for (int i = 0; i < AC; ++i) m.epret[i * N + e] = i < A ? s.ep_return[i] : 0.0f;
  }
  return upload(h, m, sl);
}

int msv_flush_stats(msv_handle* h, msv_stats* out) {
  if (!h || !out) return MSV_ERR_INVALID;
  DevGuard g(h->device);
  CK(cudaDeviceSynchronize());   // k_stats runs on stream 0: steps queued on non-blocking streams must be complete
  CK(cudaMemset(h->d_stat_reward, 0, sizeof(double) * MSV_MAX_AGENTS));
  CK(cudaMemset(h->d_stat_kills, 0, sizeof(unsigned long long) * MSV_MAX_AGENTS));
  CK(cudaMemset(h->d_stat_misc, 0, sizeof(unsigned long long) * 4));
  CK(msv_launch_stats(h->C.n_real, h->C.N, h->AC, h->S.sreward, h->S.skills, h->S.smisc, h->d_stat_reward, h->d_stat_kills, h->d_stat_misc, 0));
  h->launches++;
  double r[MSV_MAX_AGENTS]; unsigned long long k[MSV_MAX_AGENTS], mm[4];
  CK(cudaMemcpy(r, h->d_stat_reward, sizeof r, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(k, h->d_stat_kills, sizeof k, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(mm, h->d_stat_misc, sizeof mm, cudaMemcpyDeviceToHost));
  memset(out, 0, sizeof *out);
  for (int i = 0; i < MSV_MAX_AGENTS; ++i) { out->reward[i] = r[i]; out->kills[i] = (int64_t)k[i]; }
  out->steps = (int64_t)mm[0]; out->heals_used = (int64_t)mm[1]; out->boxes_placed = (int64_t)mm[2]; out->episodes = (int64_t)mm[3];
  return MSV_OK;
}

// Algorithmic HBM bytes per environment and step, per kernel (DESIGN.md "roofline numerator"): every state
// word a kernel touches in EVERY step is counted once per direction; the cold per-contact words (pseq/pimp, read
// and written only for live contacts) and the lists touched only on spawn/despawn are left out.
//   which 0: k_step   reads  agents (akin0, akin1, afat, aint, sreward, skills, epret) 76*A, boxes (box0, box1) 32*B,
//                            floor items (item0) 16*B, heals 8*H, zone (zonecur, zoneint) 32, header (hdr0, hdr1) 32,
//                            pair bit-matrices 24*PW, stats word 16, actions 6*A
//                     writes agents 76*A, zone 32, header 32, pair bit-matrices 24*PW, stats 16, camera words
//                            (obm 8, + omask 4*A when not omniscient), rewards 4*A, done 1
//   which 1: k_obs2   reads  agents (akin0, akin1, aint) 48*A, obm 8 (+ omask 4*A), hdr0 16, boxes 32*B, items 16*B,
//                            heals 8*H, zone 32 + next centre 8;   writes the observation tensors
//   which 2: k_lidar  reads  hdr0 16, boxes 32*B, items 16*B, heals 8*H, agents (akin0, akin1) 32*A;  writes 8*A*L
int64_t msv_kernel_bytes_per_env(msv_handle* h, int32_t which) {
  if (!h) return 0;
  const int64_t A = h->C.A, B = h->C.B0, H = h->C.H0, L = h->C.lidar_n, PW = h->PW;
  const int64_t om = h->C.omniscient ? 0 : 4 * A;
  if (which == 0) {
    const int64_t rd = 76 * A + 32 * B + 16 * B + 8 * H + 32 + 32 + 24 * PW + 16 + 6 * A;
    const int64_t wr = 76 * A + 32 + 32 + 24 * PW + 16 + 8 + om + 4 * A + 1;
    return rd + wr;
  }
  if (which == 1) return 48 * A + 8 + om + 16 + 32 * B + 16 * B + 8 * H + 40 + h->obs_floats * 4;
  if (which == 2) return L > 0 ? 16 + 32 * B + 16 * B + 8 * H + 32 * A + 8 * A * L : 0;
  return 0;
}
int64_t msv_bytes_per_env_step(msv_handle* h) {
  return msv_kernel_bytes_per_env(h, 0) + msv_kernel_bytes_per_env(h, 1) + msv_kernel_bytes_per_env(h, 2);
}
int64_t msv_obs_bytes_per_env(msv_handle* h) { return h ? h->obs_floats * 4 : 0; }
int64_t msv_kernel_launches(msv_handle* h) { return h ? h->launches : 0; }
int msv_tile_plan(msv_handle* h, int32_t out[4]) {
  if (!h || !out) return MSV_ERR_INVALID;
  out[0] = h->C.epb; out[1] = h->C.N / h->C.epb; out[2] = h->C.epb * h->AC; out[3] = (h->handoff && h->cfg.auto_reset != 2 && h->cfg.max_episode_steps == 0) ? 1 : 0;
  return MSV_OK;
}

/* debug: enable / read the per-phase cycle profile of k_step (not part of
 * the stable ABI; used by tests/gpu_quickbench.py) */
int msv_debug_profile(msv_handle* h, int enable, unsigned long long out[64]) {
  if (!h) return MSV_ERR_INVALID;
  DevGuard g(h->device); CK(cudaDeviceSynchronize());
  if (out) CK(msv_read_profile(out, 1));
  h->C.profile = enable;
  return MSV_OK;
}

/* debug (profile build): per-block timeline of the last k_step launch, 24 words per block */
int msv_debug_blocks(msv_handle* h, unsigned long long* out, int n_words) {
  if (!h || !out) return MSV_ERR_INVALID;
  DevGuard g(h->device); CK(cudaDeviceSynchronize());
  CK(msv_read_blocks(out, n_words));
  return MSV_OK;
}

/* debug (profile build): %globaltimer trace of the k_step -> k_obs2 hand-off of the last step, 5 rows of 4096 words */
int msv_debug_trace(msv_handle* h, unsigned long long* out, int n_words) {
  if (!h || !out) return MSV_ERR_INVALID;
  DevGuard g(h->device); CK(cudaDeviceSynchronize());
  CK(msv_read_trace(out, n_words));
  return MSV_OK;
}

void msv_philox4x32(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
  uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3], k0 = key[0], k1 = key[1];
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3; k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

}  // extern "C"
