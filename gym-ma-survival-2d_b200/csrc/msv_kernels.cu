// msv_kernels.cu -- the sm_100a kernels of libmasurv.so and their launchers.
//
// k_step  : one full MaSurvival.step (env:76-90) for every environment, a group
//           of G lanes per environment (lane g = agent g, see msv_env.cuh):
//           queue_actions -> pre_step hooks -> b2World::Step x2 -> post_step
//           hooks -> observations -> rewards -> done -> stats (-> auto-reset).
// k_reset : BaseEnv.reset (env:59-74) for every environment, or for those a mask selects.
// k_truncate: the step limit (truncated flags, finished mask) between k_step and the resets.
// k_observe: fetch_observations only (after msv_set_state).
// k_stats : flush_stats reduction.
#include "msv_env.cuh"
#include "msv_launch.h"

// debug phase profile (make PROFILE=1 + msv_debug_profile): sum over the
// leader lanes of the clock64() cycles spent in each phase of k_step
// [0..11] per-phase work sums, [12] max total, [13] its env, [16+k] phases of the slowest group,
// [32+k] time spent waiting at phase barrier k (sum), [48+k] the slowest group's waits
__device__ unsigned long long g_prof[64];
#ifdef MSV_PROFILE
// per-block timeline of the last launch: clock64() of thread 0 at kernel entry, after every phase barrier and at exit
// ([block][0] = number of stamps).  The barriers make these the block's phase durations; tests/gpu_quickbench.py --blocks
#define MSV_BLK_MAX 2048
#define MSV_BLK_STAMPS 24
// hand-off trace of the last step (%globaltimer, ns): [0] k_step block start, [1] its queue entry published,
// [2] observation tile resident, [3] its entry acquired, [4] tile written, [5] tile staged in shared memory; tests/gpu_quickbench.py --trace
#define MSV_TR_MAX 4096
#define MSV_TR_ROWS 6
__device__ unsigned long long g_tr[2 * MSV_TR_ROWS * MSV_TR_MAX];   // two steps (ticket parity), so that the gap between consecutive steps can be read
__device__ __forceinline__ unsigned long long gtime_ns() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define TRACE(row, idx) do { if (threadIdx.x == 0 && (idx) < MSV_TR_MAX) g_tr[((C.tq_ticket & 1u) * MSV_TR_ROWS + (row)) * MSV_TR_MAX + (idx)] = gtime_ns(); } while (0)
__device__ unsigned long long g_blk[MSV_BLK_MAX * MSV_BLK_STAMPS];
#define BLK_STAMP() do { if (C.profile && threadIdx.x == 0 && blockIdx.x < MSV_BLK_MAX && blk_n < MSV_BLK_STAMPS) { g_blk[blockIdx.x * MSV_BLK_STAMPS + blk_n] = (unsigned long long)clock64(); blk_n++; } } while (0)
#define PROF(k) do { if (C.profile) { long long _t = clock64(); ph[k] += (unsigned long long)(_t - t_last); t_last = _t; } } while (0)
#define PROFW(k) do { if (C.profile) { long long _t = clock64(); wt[k] += (unsigned long long)(_t - t_last); t_last = _t; } } while (0)
#else
#define PROF(k) do { } while (0)
#define PROFW(k) do { } while (0)
#define BLK_STAMP() do { } while (0)
#define TRACE(row, idx) do { } while (0)
#endif

// a cold Env member function called on a copy of the environment (see MSV_COLD in msv_env.cuh)
#define MSV_COLD_ON(env, call) do { auto c_ = env; c_.call; env.take(c_); } while (0)
// keep the warps of a block in the same phase: they then share instruction-cache lines
// Which of the ten phase barriers are kept (bit k = PHASE_SYNC(k)), per capacity class.  Measured on the stationary
// workloads with one 512-thread block per SM (profiles/r02_barriers.txt): without any barrier the step is 50 % slower
// (163 against 109 us, 2v2); dropping single ones moves it by +-1 %; for the 2- and 4-lane classes dropping the two
// between solve, FindNewContacts and SolveTOI (3 and 9: the lanes flow from the island solver into the TOI scan)
// gains 2.5 % (108.7 -> 106.0 us), while the 8-lane class is fastest with all ten (345 against 349 us).
#define MSV_SYNC_MASK(G) ((G) >= 8 ? 0x3FF : 0x1F7)
#define PHASE_SYNC(k) do { if ((MSV_SYNC_MASK(G) >> (k)) & 1) __syncthreads(); PROFW(k); BLK_STAMP(); } while (0)
// thread -> (environment slot of the block, lane of the group)
#define MSV_GROUP_SETUP(G)                                                                       \
  const int es = threadIdx.x / (G), g = threadIdx.x % (G);                                       \
  const int e = blockIdx.x * (blockDim.x / (G)) + es;  /* C.N >= gridDim.x * environments per block */ \
  const unsigned gmask = (((G) >= 32) ? 0xffffffffu : ((1u << (G)) - 1u)) << ((threadIdx.x & 31) & ~((G) - 1))

template <int AC, int BC, int HC, int G>
__global__ void __launch_bounds__(MSV_TPB)
k_step(const __grid_constant__ DevConst C, const __grid_constant__ DevState S,
       const __grid_constant__ DevOut Oc, const uint8_t* __restrict__ actions) {
  MSV_GROUP_SETUP(G);
  DevOut O = Oc;
  // Let the observation kernel (launched programmatically dependent, see msv_abi.cu launch()) become resident as
  // soon as every block of this grid has started: its blocks wait for entries of the completion queue below.
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  // Launched programmatically dependent on the previous step's observation kernel (its launch latency and block
  // start-up then overlap that kernel's tail): nothing of the state may be read or written before that grid is complete.
  if (C.pdl_wait) asm volatile("griddepcontrol.wait;" ::: "memory");
  TRACE(0, blockIdx.x);
  Env<AC, BC, HC, G> env(C, S, es, g, gmask, e);
#ifdef MSV_PROFILE
  long long t_last = C.profile ? clock64() : 0;
  const long long t_begin = t_last;
  unsigned long long ph[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  unsigned long long wt[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  int blk_n = 1;
  BLK_STAMP();
#endif
  env.load();
  const bool real = e < C.n_real;   // padding envs (N rounded up to the block size) get the no-op action
  PROF(0);
  PHASE_SYNC(0);
  const unsigned act = env.pre_motors(actions, real);   // sim:234-235; every lane reads its own agent's action
  env.gsync();
  if (env.lead) env.pre_use_give(act);
  env.gsync();
  env.share_counts();
  const int newfix = env.bc(env.LI(env.L_NEWFIX));
  if (env.bc(env.LI(env.L_NEWBOX))) env.share_bits();
  PHASE_SYNC(6);
  env.pre_melee(act);
  PROF(1);
#pragma unroll 1
  for (int sub = 0; sub < 2; ++sub) {      // sim:236-239: b2World::Step x2
    if (sub == 0 && newfix) { env.find_new_contacts(); env.LI(env.L_NEWFIX) = 0; }  // b2World::Step: e_newFixture
    PROF(2);
    PHASE_SYNC(1);
    env.collide();
    PROF(3);
    PHASE_SYNC(2);
    const int first = env.bc(env.LI(env.L_FIRST));
    env.solve(C.dt, first ? 0.0f : C.dt_ratio1);
    PROF(4);
    PHASE_SYNC(9);
    env.solve_find_new();
    PROF(2);
    PHASE_SYNC(3);
    env.solve_toi(C.dt);
    env.LI(env.L_FIRST) = 0;
    PROF(5);
  }
  if (env.lead) env.post_step_boxes();
  env.share_counts();
  PROF(6);
  PHASE_SYNC(4);
  // Cameras run on the post-physics state, before this step's deaths (env:325,330).  An environment that
  // finishes and is reset in place needs them once more for the first observation of its new episode: that
  // second evaluation goes through the SAME code (one copy of the camera / ray-cast program, already warm in
  // the instruction cache) instead of a second inlined copy that only reset environments would ever fetch.
  int again = 0;
#pragma unroll 1
  for (int pass = 0;; ++pass) {
    env.cameras();
    if (pass) break;
    PROF(7);
    PHASE_SYNC(5);
    env.post_step_rest();                  // sim:241-242
    PROF(8);
    PHASE_SYNC(7);
    if (env.lead) {
      bool done = env.rewards_done(O);     // env:85-89
      if (done && C.auto_reset) {          // vector-env extension: the observation returned is the new episode's first
        env.LI(env.L_STEPISODES)++;
        { RARE_BEGIN(); MSV_COLD_ON(env, reset()); RARE_END(2); }
        again = 1;
      }
      env.store_immune(O);
    }
    again = env.bc(again);
    if (!again) break;                     // group-uniform
    env.share_counts();
  }
  PROF(9);
  PHASE_SYNC(8);
  if (env.lead) env.store_obm();           // env:84: the observation tensors are gathered by k_obs2
  PROF(10);
  env.store();
  PROF(11);
  if (C.tq_ticket) {                       // publish this tile: every store of the block, then (release) its queue entry
    __syncthreads();
    if (threadIdx.x == 0) {           // (st.release.gpu is the fence: cumulative over the block's stores ordered before it by the barrier)
      const unsigned slot = atomicAdd(S.tq_tail, 1u) - C.tq_base;
      const unsigned long long v = ((unsigned long long)C.tq_ticket << 32) | (unsigned long long)blockIdx.x;
      asm volatile("st.release.gpu.global.u64 [%0], %1;" :: "l"(S.tq + slot), "l"(v) : "memory");
      TRACE(1, blockIdx.x);
    }
  }
#ifdef MSV_PROFILE
  __syncthreads();
  BLK_STAMP();
  if (C.profile && threadIdx.x == 0 && blockIdx.x < MSV_BLK_MAX) g_blk[blockIdx.x * MSV_BLK_STAMPS] = (unsigned long long)blk_n;
  if (C.profile && env.lead) {
    for (int k = 0; k < 12; ++k) { atomicAdd(&g_prof[k], ph[k]); atomicAdd(&g_prof[32 + k], wt[k]); }
    unsigned long long tot = (unsigned long long)(clock64() - t_begin);
    unsigned long long prev = atomicMax(&g_prof[12], tot);
    if (tot > prev) {   // (racy, indicative) phase breakdown + identity of the slowest group so far
      for (int k = 0; k < 12; ++k) { g_prof[16 + k] = ph[k]; g_prof[48 + k] = wt[k]; }
      g_prof[13] = (unsigned long long)e;
    }
  }
#endif
}

// BaseEnv.reset (env:59-74) of the environments whose byte in `mask` is set (NULL: every environment).
// finished != 0: the reset ends an episode that just finished (terminal capture, step limit): it is counted in
// flush_stats()['episodes'], and the step's outputs (rewards, dones, episode_*) stay as the step wrote them.  The
// masks of those resets (dones, k_truncate's finished mask) cover the padded batch.
// finished == 0: a restart the caller asked for (msv_reset, msv_reset_envs): not counted, and the environment's
// rewards, dones, truncated (when the handle has a step limit) and BattleRoyale flags are zeroed.  The caller's
// mask has one byte per real environment.
template <int AC, int BC, int HC, int G>
__global__ void __launch_bounds__(MSV_TPB)
k_reset(const __grid_constant__ DevConst C, const __grid_constant__ DevState S,
        const __grid_constant__ DevOut Oc, const uint8_t* __restrict__ mask, int finished, uint8_t* __restrict__ truncated) {
  MSV_GROUP_SETUP(G);
  DevOut O = Oc;
  if (mask && ((!finished && e >= C.n_real) || !mask[e])) return;    // (whole group leaves)
  Env<AC, BC, HC, G> env(C, S, es, g, gmask, e);
  env.load();
  if (env.lead) {
    if (finished) env.LI(env.L_STEPISODES)++;
    MSV_COLD_ON(env, reset());
  }
  env.share_counts();
  env.cameras();
  if (env.lead) {
    env.store_obm();
    env.store_immune(O);
    if (!finished) {
      for (int i = 0; i < C.A; ++i) O.rewards[(size_t)e * C.A + i] = 0.0f;
      O.dones[e] = 0;
      if (truncated) truncated[e] = 0;
      if (C.battle_royale) { O.br_over[e] = 0; for (int i = 0; i < C.A; ++i) O.br_results[(size_t)e * C.A + i] = 0; }   // BattleRoyale.post_reset (sem:38-39)
    }
  }
  env.store();
}

// Step limit (msv_config.max_episode_steps = T > 0), after a k_step without the in-kernel reset: an episode that
// has run T steps (hdr0.y) and did not end on this step is truncated.  Writes `truncated`, the episode_* rows of
// the truncated environments (k_step wrote those of the finished ones) and `finished` = dones | truncated, the
// rows the terminal capture keeps and the auto-reset resets.  One thread per environment of the padded batch.
__global__ void __launch_bounds__(128)
k_truncate(const __grid_constant__ DevConst C, const __grid_constant__ DevState S, const __grid_constant__ DevOut O, int T,
           uint8_t* __restrict__ truncated, uint8_t* __restrict__ finished) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= C.N) return;
  const int steps = S.hdr0[e].y;
  const bool done = O.dones[e] != 0, trunc = !done && steps >= T;
  truncated[e] = trunc ? 1 : 0;
  finished[e] = (done || trunc) ? 1 : 0;
  if (trunc) {
    for (int i = 0; i < C.A; ++i) O.episode_return[(size_t)e * C.A + i] = S.epret[i * C.N + e];
    O.episode_length[e] = steps;
  }
}

template <int AC, int BC, int HC, int G>
__global__ void __launch_bounds__(MSV_TPB)
k_observe(const __grid_constant__ DevConst C, const __grid_constant__ DevState S,
          const __grid_constant__ DevOut Oc) {
  MSV_GROUP_SETUP(G);
  Env<AC, BC, HC, G> env(C, S, es, g, gmask, e);
  env.load();
  env.cameras();
  if (env.lead) env.store_obm();
}

// fetch_observations (env:510-657), SOURCE-major: a warp takes one source item -- agent j, box k,
// floor item k, heal k, the zone -- for 32 consecutive environments (lane = environment: the SoA
// loads are fully coalesced), builds everything that item contributes (an agent row goes to `agent`
// and to the `others` block of every other observer; observer j's mask rows and inventory-slot views)
// and scatters it into a shared-memory stage laid out exactly like the 32-environment slice of each
// output tensor.  The stage is then copied out with 16-byte stores, one contiguous run per tensor.
// kRows (terminal capture): only the rows of real environments whose `only_if` byte is set are
// written, with scalar stores (a row's slice of a key is not 16-byte aligned in general); the other
// rows of the output are left untouched, and a tile without such a row leaves at once.
// kFlat (MSV_OBS_FLAT): the stage keeps the layout above (a stage in the flat layout, with the keys stored once
// per environment repeated for every agent, would not fit in shared memory for 8 agents); only the copy-out
// changes.  The tile's rows of obs_flat are ONE contiguous run of rows * A * D floats, 16-byte aligned (e0 and
// rows are multiples of 4), written with 16-byte stores, each float gathered from the stage through the
// per-column map F.map (held in shared memory after the stage).  A float4 that holds only lidar columns is not
// written (k_lidar writes them after this kernel); one that straddles them writes stage[0] there.
template <bool kRows, bool kFlat>
__global__ void __launch_bounds__(1024)
k_obs2(const __grid_constant__ DevConst C, const __grid_constant__ DevState S, const __grid_constant__ ObsTable Tb, int AC,
       const uint8_t* __restrict__ only_if, const ObsFlat F) {
  extern __shared__ float stage[];
  const int A = C.A, B = C.B0, H = C.H0, Sw = C.S, N = C.N;
  // A tile is (part of) the environments of one k_step block: block `kb`, sub-tile `sub` of up to OBS2_E rows.
  // With the hand-off on (C.tq_ticket != 0) `kb` is the (blockIdx.x / spb)-th block of the running step kernel
  // to finish, read from its completion queue; otherwise tiles are taken in index order.
  const int spb = (C.epb + OBS2_E - 1) / OBS2_E;
  int kb = blockIdx.x / spb; const int sub = blockIdx.x - kb * spb;
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  TRACE(2, blockIdx.x);
  if (!kRows && C.tq_ticket) {                   // (a row-filtered launch is never part of a hand-off)
    __shared__ int s_kb;
    if (threadIdx.x == 0) {
      const unsigned long long* q = S.tq + kb;
      unsigned long long v;
      int spins = 0;
      // Poll with relaxed loads and fence once at the end: an acquire load is LDG.STRONG + CCTL.IVALL, and
      // invalidating the SM's L1 on every poll would take the local-memory lines of the step-kernel block that
      // shares the SM with it.
      for (;;) {
        asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(q) : "memory");
        if ((unsigned)(v >> 32) == C.tq_ticket) break;
        // (never seen: ~4 s without the entry -> record a fault for msv_debug_overflow and take the tile by index, so
        // that a broken hand-off shows up as a failing test instead of a hung device)
        if (++spins > (1 << 22)) { S.tq_tail[2] = 1u; v = (unsigned long long)kb; break; }
        __nanosleep(1000);
      }
      asm volatile("fence.acq_rel.gpu;" ::: "memory");
      s_kb = (int)(unsigned)(v & 0xffffffffull);
    }
    __syncthreads();
    kb = s_kb;
  }
  TRACE(3, blockIdx.x);
  const int e0 = kb * C.epb + sub * OBS2_E, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int rows = C.epb - sub * OBS2_E; if (rows > OBS2_E) rows = OBS2_E;   // a multiple of 32 / G >= 4: every run below is a whole number of float4
  // this lane's row of every tensor slice in the stage (registers: the key is a compile-time constant at every use)
  int koff[MSV_OBS_KEYS], kbase[MSV_OBS_KEYS], stage_floats = 0;
  {
    int o = 0;
#pragma unroll
    for (int k = 0; k < MSV_OBS_KEYS; ++k) { koff[k] = o; kbase[k] = o + lane * Tb.keys[k].chunk; o += OBS2_E * Tb.keys[k].chunk; }
    stage_floats = o;
  }
  const int e = e0 + lane;
  const bool live = lane < rows;                 // (e < N: the padded batch is a whole number of k_step blocks)
  unsigned sel = 0u;                             // kRows: bit r = row r is written (every warp computes the same mask)
  if (kRows) {
    sel = __ballot_sync(0xffffffffu, live && e < C.n_real && only_if[e] != 0);
    if (!sel) return;
  }
  int2* fmap = reinterpret_cast<int2*>(stage + stage_floats);
  if (kFlat)
    for (int c = threadIdx.x; c < F.D; c += blockDim.x) fmap[c] = __ldg(&F.map[c]);
  const int n_items = A + 2 * B + H + 1;
  // (state loads below bypass L1 -- __ldcg: each word is read once, and with the hand-off on it was written by a
  // block of the still-running step kernel on another SM)
  auto put = [&](int key, int off, float v) { stage[kbase[key] + off] = v; };
  auto vert = [&](float hx, float hy, int rot, int comp) {   // b2PolygonShape vertex order (Q8)
    int j = ((comp >> 1) + rot) & 3;
    return (comp & 1) ? ((j >= 2) ? hy : -hy) : ((j == 1 || j == 2) ? hx : -hx);
  };
  const int nwarps = blockDim.x >> 5;
  for (int it = warp; it < n_items; it += nwarps) {
    if (it < A) {                                // ---- agent j: its row everywhere + observer j's own views
      const int j = it;
      int inv = 0; bool al = false; unsigned long long obm = 0ull; unsigned om = 0u; int cnts = 0;
      float4 pl = make_float4(0.f, 0.f, 0.f, 0.f);
      float r_id = 0.f, r_team = 0.f, r_hp = 0.f, r_x = 0.f, r_y = 0.f, r_a = 0.f, r_vx = 0.f, r_vy = 0.f, r_w = 0.f;   // env:659-691
      if (live) {
        const float4 k0 = __ldcg(&S.akin0[j * N + e]), k1 = __ldcg(&S.akin1[j * N + e]); const int4 ai = __ldcg(&S.aint[j * N + e]);
        al = (__float_as_int(k1.w) & 1) != 0; inv = ai.w; obm = __ldcg(&S.obm[e]); cnts = __ldcg(&S.hdr0[e].x);
        if (!C.omniscient) om = __ldcg(&S.omask[j * N + e]);
        r_id = (float)j; r_team = (float)(j < A / 2 ? 0 : 1);
        if (al) { r_hp = (float)ai.x; r_x = k0.x; r_y = k0.y; r_a = k0.z; r_vx = k0.w; r_vy = k1.x; r_w = k1.y; }
        const int n = inv & 7;
        if (al && n > 0 && ((inv >> (4 + 2 * (n - 1))) & 3) == MSV_ITEM_BOX) pl = __ldcg(&S.ainv[(j * 4 + n - 1) * N + e]);
      }
      const int tm = C.teams ? 1 : 0;
      auto emit = [&](int key, int base) {         // [id, (team), health, x, y, angle, vx, vy, omega]
        put(key, base, r_id); if (tm) put(key, base + 1, r_team);
        put(key, base + tm + 1, r_hp); put(key, base + tm + 2, r_x); put(key, base + tm + 3, r_y); put(key, base + tm + 4, r_a);
        put(key, base + tm + 5, r_vx); put(key, base + tm + 6, r_vy); put(key, base + tm + 7, r_w);
      };
      emit(0, j * Sw);
      for (int i = 0; i < A; ++i) {              // others[i][k]: agents in index order skipping the observer (env:529-534)
        if (i == j) continue;
        emit(1, (i * (A - 1) + (j < i ? j : j - 1)) * Sw);
      }
      for (int q = 0; q < A; ++q) {              // others_mask[j][k]: 0 = seen by observer j's camera (env:692-703)
        if (q == j) continue;
        const int k = q < j ? q : q - 1;
        put(2, j * (A - 1) + k, ((obm >> (j * AC + q)) & 1ull) ? 0.0f : 1.0f);
      }
      const int nb = cnts & 255, ni = (cnts >> 8) & 255, nh = (cnts >> 16) & 255;
      const int n = inv & 7; const int top = n > 0 ? (inv >> (4 + 2 * (n - 1))) & 3 : 0;
      if (H > 0) {
        for (int k = 0; k < H; ++k) {
          const bool seen = C.omniscient ? k < nh : (k < nh && al && ((om >> k) & 1u));      // env:564-568 / 706-739
          put(5, j * H + k, (live && seen) ? 0.0f : 1.0f);
        }
        const bool has = al && top == MSV_ITEM_HEAL;
        put(6, j, has ? (float)C.healing : 0.0f); put(7, j, has ? 0.0f : 1.0f);
      }
      if (B > 0) {
        for (int k = 0; k < B; ++k) {
          const bool sb_ = C.omniscient ? k < nb : (k < nb && al && ((om >> (16 + k)) & 1u));
          const bool si_ = C.omniscient ? k < ni : (k < ni && al && ((om >> (24 + k)) & 1u));
          put(9, j * B + k, (live && sb_) ? 0.0f : 1.0f); put(11, j * B + k, (live && si_) ? 0.0f : 1.0f);
        }
        const bool has = al && top == MSV_ITEM_BOX;
        for (int c = 0; c < 8; ++c) put(12, j * 8 + c, has ? vert(pl.x, pl.y, __float_as_int(pl.w) & 1, c) : 0.0f);
        put(13, j, has ? 0.0f : 1.0f);
      }
    } else if (it < A + B) {                     // ---- box k (env:570-591)
      const int k = it - A;
      float4 b0 = make_float4(0.f, 0.f, 0.f, 0.f); int rot = 0; bool on = false;
      if (live && k < (__ldcg(&S.hdr0[e].x) & 255)) { b0 = __ldcg(&S.box0[k * N + e]); rot = (__ldcg(&S.box1[k * N + e].y) >> 1) & 1; on = true; }
      for (int c = 0; c < 8; ++c) put(8, k * 11 + c, on ? vert(b0.z, b0.w, rot, c) : 0.0f);
      put(8, k * 11 + 8, on ? b0.x : 0.0f); put(8, k * 11 + 9, on ? b0.y : 0.0f); put(8, k * 11 + 10, 0.0f);
    } else if (it < A + 2 * B) {                 // ---- floor box item k (env:593-619)
      const int k = it - A - B;
      float4 i0 = make_float4(0.f, 0.f, 0.f, 0.f); bool on = false;
      if (live && k < ((__ldcg(&S.hdr0[e].x) >> 8) & 255)) { i0 = __ldcg(&S.item0[k * N + e]); on = true; }
      for (int c = 0; c < 8; ++c) put(10, k * 10 + c, on ? vert(i0.z, i0.w, 1, c) : 0.0f);
      put(10, k * 10 + 8, on ? i0.x : 0.0f); put(10, k * 10 + 9, on ? i0.y : 0.0f);
    } else if (it < A + 2 * B + H) {             // ---- heal k (env:552-568)
      const int k = it - A - 2 * B;
      float2 hh = make_float2(0.f, 0.f);
      if (live && k < ((__ldcg(&S.hdr0[e].x) >> 16) & 255)) hh = __ldcg(&S.heal[k * N + e]);
      put(4, 2 * k, hh.x); put(4, 2 * k + 1, hh.y);
    } else {                                     // ---- zone (env:537-550)
      float z[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      if (live) {
        const float4 zc = __ldcg(&S.zonecur[e]); const int ph = __ldcg(&S.zoneint[e].x);
        z[0] = zc.x; z[1] = zc.y; z[2] = zc.z;
        if (ph < C.zone_phases - 1) { const float2 c2 = __ldcg(&S.zonec[(ph + 1) * N + e]); z[3] = c2.x; z[4] = c2.y; z[5] = C.zone_r32[ph + 1]; }
      }
      for (int c = 0; c < 6; ++c) put(3, c, z[c]);
    }
  }
  __syncthreads();
  TRACE(5, blockIdx.x);
  if (kFlat) {
    const int D = F.D, AD = A * D, DL = D - C.lidar_n;
    float* dst = F.base + (size_t)e0 * AD;
    auto gather = [&](int r, int i, int c) { const int2 m = fmap[c]; return stage[m.x + r * (m.y & 0xffff) + i * (m.y >> 16)]; };
    if (kRows) {
      for (int q = threadIdx.x; q < rows * AD; q += blockDim.x) {
        const int r = q / AD, rem = q - r * AD, i = rem / D, c = rem - i * D;
        if (((sel >> r) & 1u) && c < DL) dst[q] = gather(r, i, c);
      }
    } else {
      float4* dst4 = reinterpret_cast<float4*>(dst);
      for (int q4 = threadIdx.x; q4 < rows * AD / 4; q4 += blockDim.x) {
        const int q = 4 * q4;
        int r = q / AD; const int rem = q - r * AD; int i = rem / D; int c = rem - i * D;
        if (c >= DL && c + 3 < D) continue;      // four lidar columns of one agent's row
        float v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          v[u] = gather(r, i, c);
          if (++c == D) { c = 0; if (++i == A) { i = 0; ++r; } }
        }
        dst4[q4] = make_float4(v[0], v[1], v[2], v[3]);
      }
    }
  } else {
    for (int k = 0; k < MSV_OBS_KEYS; ++k) {
      const int chunk = Tb.keys[k].chunk;
      if (chunk <= 0 || !obs_key_used(k, H, B)) continue;
      if (kRows) {
        const float* src = stage + koff[k];
        float* dst = Tb.keys[k].base + (size_t)e0 * chunk;
        for (int q = threadIdx.x; q < rows * chunk; q += blockDim.x)
          if ((sel >> (q / chunk)) & 1u) dst[q] = src[q];
      } else {
        const int n4 = rows * chunk / 4;
        const float4* src = reinterpret_cast<const float4*>(stage + koff[k]);
        float4* dst = reinterpret_cast<float4*>(Tb.keys[k].base + (size_t)e0 * chunk);
        for (int q = threadIdx.x; q < n4; q += blockDim.x) dst[q] = src[q];
      }
    }
  }
  TRACE(4, blockIdx.x);
  if (!kRows && C.tq_ticket) {
    // The last tile to finish waits for the step kernel's grid to have completed, so that "this grid is complete"
    // implies "the step kernel is complete" for whatever follows in the stream, whichever way the runtime orders
    // a third kernel after a programmatic pair.  (Every other block has already seen its tile's release.)
    __syncthreads();
    if (threadIdx.x == 0) {
      const unsigned d = atomicAdd(S.tq_tail + 1, 1u);
      if (d == gridDim.x - 1) { S.tq_tail[1] = 0u; asm volatile("griddepcontrol.wait;" ::: "memory"); }
    }
  }
}

// Lidars._update (simulation.py:377-392) as an extension observation block, scanned on the state the
// observation describes.  ONE WARP PER AGENT, rays across the lanes.  A block covers whole environments:
// it first stages the environment's bodies (scan order: boxes, box items, heals, walls, agents) as a
// table in shared memory; each warp then culls the table against its agent's fan -- one body per lane,
// range and (for fans narrower than a half plane) the two edge half-planes, conservatively -- and the
// surviving bodies are ray-tested by every lane.  The minimum fraction wins; of equal fractions the body
// created first (smallest body sequence number) wins, as in the oracle's scan of the world's body list.
#define LID_MAXB 64            // >= MSV_MAX_BOXES * 2 + MSV_MAX_HEALS + 4 + MSV_MAX_AGENTS = 44
#define LID_W 9
__global__ void __launch_bounds__(256)
k_lidar(const __grid_constant__ DevConst C, const __grid_constant__ DevState S, const __grid_constant__ DevOut O, int EB, int BC, int HC,
        int LS) {
  extern __shared__ float lid_sm[];                  // [EB][LID_MAXB][LID_W]: kind, x, y, then r | hx, hy, ax, ay, rot (agents: r, angle); [8] body seq
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // (the next step's k_step may be waiting to become resident)
  const int A = C.A, L = C.lidar_n, N = C.N;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int el = warp / A, i = warp - el * A;        // environment slot of the block, agent
  const int e = blockIdx.x * EB + el;
  const bool on = e < C.n_real;
  // table slots are the CAPACITY slots of every list (boxes, box items, heals, walls, agents: the scan order), so
  // that no load depends on the list lengths: slots past a list's length become KIND_NONE.  One memory round trip.
  const int oI = BC, oH = 2 * BC, oW = 2 * BC + HC, oA = oW + 4, T = oA + A;
  float* tab = lid_sm + (size_t)el * LID_MAXB * LID_W;
  if (on) {
    const int c = S.hdr0[e].x;
    const int nb = c & 255, ni = (c >> 8) & 255, nh = (c >> 16) & 255;
    for (int b = i * 32 + lane; b < T; b += A * 32) {
      float* t = tab + b * LID_W;
      if (b < oI) {
        const float4 b0 = S.box0[b * N + e]; const int reh = (S.box1[b * N + e].y >> 1) & 1;
        SBox bx; sb_set_shape(bx, b0.z, b0.w, reh);
        t[0] = __int_as_float(b < nb ? KIND_BOX : KIND_NONE); t[1] = b0.x; t[2] = b0.y; t[3] = bx.hx; t[4] = bx.hy; t[5] = bx.ax; t[6] = bx.ay; t[7] = __int_as_float(bx.rot);
        t[8] = __int_as_float(S.boxseq[b * N + e]);
      } else if (b < oH) {
        const float4 it = S.item0[(b - oI) * N + e];
        t[0] = __int_as_float(b - oI < ni ? KIND_ITEM : KIND_NONE); t[1] = it.x; t[2] = it.y; t[3] = C.item_r;
        t[8] = __int_as_float(S.item1[(b - oI) * N + e].y);
      } else if (b < oW) {
        const float2 hh = S.heal[(b - oH) * N + e];
        t[0] = __int_as_float(b - oH < nh ? KIND_HEAL : KIND_NONE); t[1] = hh.x; t[2] = hh.y; t[3] = C.heal_r;
        t[8] = __int_as_float(S.healseq[(b - oH) * N + e]);
      } else if (b < oA) {
        t[0] = __int_as_float(KIND_WALL); t[1] = C.walls[b - oW].px; t[2] = C.walls[b - oW].py; t[3] = __int_as_float(b - oW);
        t[8] = __int_as_float(C.B0 + C.H0 + (b - oW));     // the walls and agents keep the sequence numbers of the reset
      } else {
        const float4 o = S.akin0[(b - oA) * N + e];
        const bool al = (__float_as_int(S.akin1[(b - oA) * N + e].w) & 1) != 0;
        t[0] = __int_as_float(al ? KIND_AGENT : KIND_NONE); t[1] = o.x; t[2] = o.y; t[3] = C.agent_r; t[4] = o.z;
        t[8] = __int_as_float(C.B0 + C.H0 + 4 + (b - oA));
      }
    }
  }
  __syncthreads();
  if (!on) return;
  const float* mine = tab + (oA + i) * LID_W;
  const bool alive_i = __float_as_int(mine[0]) == KIND_AGENT;
  const size_t obase = ((size_t)e * A + i) * L, fbase = ((size_t)e * A + i) * LS;   // lidar_frac rows: LS apart (flat layout: D)
  if (!alive_i) {                                    // dead agents have no Lidars row: reported as "no hit"
    if (lane < L) { O.lidar_frac[fbase + lane] = 1.0f; O.lidar_hit[obase + lane] = 0; }
    return;
  }
  const f2 me = mk2(mine[1], mine[2]);
  const float heading = mine[4];
  // ---- cull: which bodies can any ray of this fan reach?  (conservative; never the agent itself)
  unsigned long long cand = 0ull;
  {
    const float hf = 0.5f * (float)(C.lidar_ang[L - 1] - C.lidar_ang[0]);          // half the fan
    const bool convex = L > 1 && hf < 1.45f;                                       // fan inside a half plane (with margin)
    float sl, cl, sr, cr;
    sincosf(heading + hf, &sl, &cl); sincosf(heading - hf, &sr, &cr);
#pragma unroll
    for (int round = 0; round < LID_MAXB / 32; ++round) {
      const int b = round * 32 + lane;
      bool keep = false;
      if (b < T) {
        const float* t = tab + b * LID_W;
        const int kind = __float_as_int(t[0]);
        if (kind == KIND_WALL) keep = true;                                        // long thin boxes: the per-ray test handles them
        else if (kind != KIND_NONE && b != oA + i) {
          const float bound = kind == KIND_BOX ? t[3] + t[4] + 0.02f : t[3] + 0.02f;    // |hx|+|hy| >= circumradius
          const float dx = t[1] - me.x, dy = t[2] - me.y;
          const float dist = sqrtf(dx * dx + dy * dy);
          const float slack = bound + 1e-3f * (1.0f + dist);
          keep = dist <= C.lidar_depth + slack;
          if (keep && convex && dist > slack) {
            const float crossL = cl * dy - sl * dx, crossR = cr * dy - sr * dx;    // > 0: left of that edge
            if (crossL > slack || crossR < -slack) keep = false;
          }
        }
      }
      const unsigned m = __ballot_sync(0xffffffffu, keep);
      cand |= (unsigned long long)m << (32 * round);
    }
  }
  // ---- rays
  if (lane < L) {
    const int r = lane;
    const double ang = C.lidar_ang[r] + (double)heading;
    const f2 off = from_polar(C.lidar_depth, (float)ang);
    const f2 p2 = vadd(me, off);
    const float lx = fmin_(me.x, p2.x), ly = fmin_(me.y, p2.y), ux = fmax_(me.x, p2.x), uy = fmax_(me.y, p2.y);
    // conservative reject before every exact test: distance from the body's centre to the ray's segment against a
    // bound of the shape (much tighter than the segment's AABB for a 10 m ray); it can only skip shapes the exact test would miss
    const float dd = C.lidar_depth;
    auto far_from = [&](float cx, float cy, float rad) {
      const float dx = cx - me.x, dy = cy - me.y, lim = (rad + 0.01f) * dd;
      const float perp = off.x * dy - off.y * dx, along = off.x * dx + off.y * dy;
      return fabsf(perp) > lim || along < -lim || along > dd * dd + lim;
    };
    float best = 2.0f; int bestb = -1, bestseq = 0;
    unsigned long long m = cand;
    while (m) {
      const int b = __ffsll((long long)m) - 1; m &= m - 1;
      const float* t = tab + b * LID_W;
      const int kind = __float_as_int(t[0]);
      float f; bool hit = false;
      if (kind == KIND_BOX) {
        if (!far_from(t[1], t[2], t[3] + t[4] + 0.01f)) {
          SBox bx; bx.px = t[1]; bx.py = t[2]; bx.qs = 0.0f; bx.qc = 1.0f; bx.ang = 0.0f;
          bx.hx = t[3]; bx.hy = t[4]; bx.ax = t[5]; bx.ay = t[6]; bx.rot = __float_as_int(t[7]);
          hit = ray_box(bx, me, p2, f);
        }
      } else if (kind == KIND_WALL) {
        const WallC& w = C.walls[__float_as_int(t[3])];
        if (!(w.fat[2] < lx || w.fat[0] > ux || w.fat[3] < ly || w.fat[1] > uy)) {
          SBox bx; bx.px = w.px; bx.py = w.py; bx.qs = w.qs; bx.qc = w.qc; bx.ang = w.ang; bx.hx = C.wall_hx; bx.hy = C.wall_hy; bx.ax = 1.0f; bx.ay = 1.0f; bx.rot = 0;
          hit = ray_box(bx, me, p2, f);
        }
      } else {                                         // item, heal or agent circle
        if (!far_from(t[1], t[2], t[3] + 0.01f)) hit = ray_circle(mk2(t[1], t[2]), t[3], me, p2, f);
      }
      if (hit && (f < best || (f == best && __float_as_int(t[8]) < bestseq))) { best = f; bestb = b; bestseq = __float_as_int(t[8]); }
    }
    float fr = 1.0f; int hitcode = 0;
    if (bestb >= 0) {
      fr = best;
      int kind, idx;
      if (bestb < oI) { kind = KIND_BOX; idx = bestb; }
      else if (bestb < oH) { kind = KIND_ITEM; idx = bestb - oI; }
      else if (bestb < oW) { kind = KIND_HEAL; idx = bestb - oH; }
      else if (bestb < oA) { kind = KIND_WALL; idx = bestb - oW; }
      else { kind = KIND_AGENT; idx = bestb - oA; }
      hitcode = (kind << 8) | idx;
    }
    O.lidar_frac[fbase + r] = fr;
    O.lidar_hit[obase + r] = hitcode;
  }
}

// Pre-draw the reset record of every environment whose record is not the one of its NEXT episode (after a
// reset, after msv_set_state).  Runs beside the observation kernels, off the step kernel's critical path: the
// in-kernel reset of a finished environment then only copies 96 floats instead of running the Philox shuffle,
// the Box-Muller box shapes and the zone-centre draws while the 63 other environments of its block wait.
// `only_done`: look only at the environments whose done flag is set (the ones the step just reset).
__global__ void __launch_bounds__(128)
k_spare(const __grid_constant__ DevConst C, const __grid_constant__ DevState S, const uint8_t* __restrict__ dones, int only_done) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= C.n_real) return;
  if (only_done && !dones[e]) return;
  const int next = S.hdr0[e].z + 1;
  if (S.spare_ep[e] == next) return;
  float rec[MSV_SPARE_W];
#pragma unroll
  for (int q = 0; q < MSV_SPARE_W; ++q) rec[q] = 0.0f;
  draw_reset(C, C.env_offset + (uint32_t)e, (uint32_t)next, rec);
  float4* dst = reinterpret_cast<float4*>(S.spare + (size_t)e * MSV_SPARE_W);
#pragma unroll
  for (int q = 0; q < MSV_SPARE_W / 4; ++q) dst[q] = make_float4(rec[4 * q], rec[4 * q + 1], rec[4 * q + 2], rec[4 * q + 3]);
  __threadfence();
  S.spare_ep[e] = next;
}

cudaError_t msv_launch_spare(const DevConst& C, const DevState& S, const uint8_t* dones, int only_done, cudaStream_t st) {
  k_spare<<<(C.n_real + 127) / 128, 128, 0, st>>>(C, S, dones, only_done);
  return cudaPeekAtLastError();
}

// flush_stats (env:471-480): sum the per-env accumulators, then zero them
__global__ void k_stats(int N, int stride, int AC, float* sreward, int* skills, int4* smisc,
                        double* out_reward, unsigned long long* out_kills, unsigned long long* out_misc) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  double r[MSV_MAX_AGENTS]; long long k[MSV_MAX_AGENTS]; long long m[4] = {0, 0, 0, 0};
  for (int i = 0; i < MSV_MAX_AGENTS; ++i) { r[i] = 0.0; k[i] = 0; }
  if (e < N) {
    for (int i = 0; i < AC; ++i) {
      r[i] = sreward[i * stride + e]; k[i] = skills[i * stride + e];
      sreward[i * stride + e] = 0.0f; skills[i * stride + e] = 0;
    }
    int4 s = smisc[e]; m[0] = s.x; m[1] = s.y; m[2] = s.z; m[3] = s.w;
    smisc[e] = make_int4(0, 0, 0, 0);
  }
  for (int off = 16; off > 0; off >>= 1) {
    for (int i = 0; i < AC; ++i) { r[i] += __shfl_down_sync(0xffffffffu, r[i], off); k[i] += __shfl_down_sync(0xffffffffu, k[i], off); }
    for (int i = 0; i < 4; ++i) m[i] += __shfl_down_sync(0xffffffffu, m[i], off);
  }
  if ((threadIdx.x & 31) == 0) {
    for (int i = 0; i < AC; ++i) { atomicAdd(&out_reward[i], r[i]); atomicAdd(&out_kills[i], (unsigned long long)k[i]); }
    for (int i = 0; i < 4; ++i) atomicAdd(&out_misc[i], (unsigned long long)m[i]);
  }
}

// ------------------------------------------------------------- launchers ---
template <bool kRows, bool kFlat>
static cudaError_t obs_attrs() {
  // the stage of the 8-agent class is ~1 000 floats x 32 environments, far over the 48 KB default
  cudaError_t e = cudaFuncSetAttribute(k_obs2<kRows, kFlat>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  // same L1/shared split as the step kernel, so that a tile can become resident on an SM that still runs one of its blocks
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(k_obs2<kRows, kFlat>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  return e;
}

template <int AC, int BC, int HC, int G>
static cudaError_t launch_t(int which, const DevConst& C, const DevState& S, const DevOut& O,
                            const uint8_t* actions, cudaStream_t st) {
  const int epb = C.epb;                             // environments per block (runtime: msv_plan_blocks)
  const int blocks = C.N / epb, tpb = epb * G;
  size_t smem = (size_t)Env<AC, BC, HC, G>::SM_WORDS * epb * sizeof(float);
  size_t smem_max = (size_t)Env<AC, BC, HC, G>::SM_WORDS * (MSV_TPB / G) * sizeof(float);
  if (smem_max > 227 * 1024) smem_max = 227 * 1024;   // (plan_blocks keeps the tile within the per-block limit)
  if (which == 3) {  // one-time, on the handle's device: allow the dynamic shared memory the kernels need
    cudaError_t e = cudaFuncSetAttribute(k_step<AC, BC, HC, G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_reset<AC, BC, HC, G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_observe<AC, BC, HC, G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max);
    if (e == cudaSuccess) e = obs_attrs<false, false>();
    if (e == cudaSuccess) e = obs_attrs<true, false>();
    if (e == cudaSuccess) e = obs_attrs<false, true>();
    if (e == cudaSuccess) e = obs_attrs<true, true>();
    return e;
  }
  if (which == 0 && C.pdl_wait) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)blocks); cfg.blockDim = dim3((unsigned)tpb); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, k_step<AC, BC, HC, G>, C, S, O, actions);
  }
  if (which == 0) k_step<AC, BC, HC, G><<<blocks, tpb, smem, st>>>(C, S, O, actions);
  else k_observe<AC, BC, HC, G><<<blocks, tpb, smem, st>>>(C, S, O);
  return cudaPeekAtLastError();
}

template <int AC, int BC, int HC, int G>
static cudaError_t reset_t(const DevConst& C, const DevState& S, const DevOut& O, const uint8_t* mask, int finished,
                           uint8_t* truncated, cudaStream_t st) {
  const size_t smem = (size_t)Env<AC, BC, HC, G>::SM_WORDS * C.epb * sizeof(float);
  k_reset<AC, BC, HC, G><<<C.N / C.epb, C.epb * G, smem, st>>>(C, S, O, mask, finished, truncated);
  return cudaPeekAtLastError();
}

cudaError_t msv_launch(int cap, int which, const DevConst& C, const DevState& S, const DevOut& O,
                       const uint8_t* actions, cudaStream_t st) {
  switch (cap) {
    case 0: return launch_t<2, 4, 4, 2>(which, C, S, O, actions, st);
    case 1: return launch_t<4, 4, 4, 4>(which, C, S, O, actions, st);
    default: return launch_t<8, 8, 16, 8>(which, C, S, O, actions, st);
  }
}

cudaError_t msv_launch_reset(int cap, const DevConst& C, const DevState& S, const DevOut& O, const uint8_t* mask, int finished,
                             uint8_t* truncated, cudaStream_t st) {
  switch (cap) {
    case 0: return reset_t<2, 4, 4, 2>(C, S, O, mask, finished, truncated, st);
    case 1: return reset_t<4, 4, 4, 4>(C, S, O, mask, finished, truncated, st);
    default: return reset_t<8, 8, 16, 8>(C, S, O, mask, finished, truncated, st);
  }
}

cudaError_t msv_launch_truncate(const DevConst& C, const DevState& S, const DevOut& O, int T, uint8_t* truncated, uint8_t* finished,
                                cudaStream_t st) {
  k_truncate<<<(C.N + 127) / 128, 128, 0, st>>>(C, S, O, T, truncated, finished);
  return cudaPeekAtLastError();
}

cudaError_t msv_launch_obs(const DevConst& C, const DevState& S, const ObsTable& T, const ObsFlat* F, int AC, const uint8_t* only_if,
                           cudaStream_t st) {
  size_t smem = 0;
  for (int k = 0; k < MSV_OBS_KEYS; ++k) smem += (size_t)OBS2_E * T.keys[k].chunk * sizeof(float);
  if (F) smem += (size_t)F->D * sizeof(int2);                          // the column map
  // one warp per source item when they fit a block (a single round of loads), else 32 warps looping over the items
  const int n_items = C.A + 2 * C.B0 + C.H0 + 1;
  const int threads = n_items <= 32 ? 32 * n_items : 1024;
  const int spb = (C.epb + OBS2_E - 1) / OBS2_E;                       // tiles per k_step block
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)((C.N / C.epb) * spb)); cfg.blockDim = dim3((unsigned)threads);
  cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;                // may start before the step kernel has finished
  cfg.attrs = at; cfg.numAttrs = C.tq_ticket ? 1 : 0;
  const ObsFlat none = {nullptr, nullptr, 0};
  if (F && only_if) return cudaLaunchKernelEx(&cfg, k_obs2<true, true>, C, S, T, AC, only_if, *F);
  if (F) return cudaLaunchKernelEx(&cfg, k_obs2<false, true>, C, S, T, AC, only_if, *F);
  if (only_if) return cudaLaunchKernelEx(&cfg, k_obs2<true, false>, C, S, T, AC, only_if, none);
  return cudaLaunchKernelEx(&cfg, k_obs2<false, false>, C, S, T, AC, only_if, none);
}

cudaError_t msv_launch_lidar(const DevConst& C, const DevState& S, const DevOut& O, int BC, int HC, int LS, cudaStream_t st) {
  int EB = 8 / C.A; if (EB < 1) EB = 1;              // whole environments per block, 8 warps (A = 8: one env; A = 4: two; A <= 2: four)
  const int warps = EB * C.A;
  const size_t smem = (size_t)EB * LID_MAXB * LID_W * sizeof(float);
  k_lidar<<<(C.n_real + EB - 1) / EB, warps * 32, smem, st>>>(C, S, O, EB, BC, HC, LS);
  return cudaPeekAtLastError();
}

void msv_capacity(int cap, int* AC, int* BC, int* HC, int* P, int* PW, int* sm_words) {
  switch (cap) {
    case 0: *AC = 2; *BC = 4; *HC = 4; *P = PairLayout<2, 4>::P; *PW = PairLayout<2, 4>::PW; *sm_words = Env<2, 4, 4, 2>::SM_WORDS; break;
    case 1: *AC = 4; *BC = 4; *HC = 4; *P = PairLayout<4, 4>::P; *PW = PairLayout<4, 4>::PW; *sm_words = Env<4, 4, 4, 4>::SM_WORDS; break;
    default: *AC = 8; *BC = 8; *HC = 16; *P = PairLayout<8, 8>::P; *PW = PairLayout<8, 8>::PW; *sm_words = Env<8, 8, 16, 8>::SM_WORDS; break;
  }
}

cudaError_t msv_launch_stats(int N, int stride, int AC, float* sreward, int* skills, int4* smisc, double* out_reward,
                             unsigned long long* out_kills, unsigned long long* out_misc, cudaStream_t st) {
  k_stats<<<(N + 127) / 128, 128, 0, st>>>(N, stride, AC, sreward, skills, smisc, out_reward, out_kills, out_misc);
  return cudaPeekAtLastError();
}

cudaError_t msv_read_check(unsigned long long out[2]) {
#ifdef MSV_CHECK
  return cudaMemcpyFromSymbol(out, g_chk, sizeof(unsigned long long) * 2);
#else
  out[0] = ~0ull; out[1] = 0;      // not a checked build
  return cudaSuccess;
#endif
}

cudaError_t msv_read_blocks(unsigned long long* out, int n_words) {   // development: the per-block timeline of the last k_step launch
#ifdef MSV_PROFILE
  if (n_words > MSV_BLK_MAX * MSV_BLK_STAMPS) n_words = MSV_BLK_MAX * MSV_BLK_STAMPS;
  cudaError_t e_ = cudaMemcpyFromSymbol(out, g_blk, sizeof(unsigned long long) * (size_t)n_words);
  if (e_ == cudaSuccess && n_words >= MSV_BLK_MAX * MSV_BLK_STAMPS) {   // the last row: the longest solve_toi call (g_toi), then cleared
    e_ = cudaMemcpyFromSymbol(out + (MSV_BLK_MAX - 1) * MSV_BLK_STAMPS, g_toi, sizeof(unsigned long long) * 16);
    unsigned long long z[16] = {0}; cudaMemcpyToSymbol(g_toi, z, sizeof z);
  }
  return e_;
#else
  (void)out; (void)n_words; return cudaErrorNotSupported;
#endif
}

cudaError_t msv_read_trace(unsigned long long* out, int n_words) {     // development: hand-off trace of the last step
#ifdef MSV_PROFILE
  if (n_words > 2 * MSV_TR_ROWS * MSV_TR_MAX) n_words = 2 * MSV_TR_ROWS * MSV_TR_MAX;
  cudaError_t e_ = cudaMemcpyFromSymbol(out, g_tr, sizeof(unsigned long long) * (size_t)n_words);
  if (e_ == cudaSuccess) { static unsigned long long z[2 * MSV_TR_ROWS * MSV_TR_MAX]; e_ = cudaMemcpyToSymbol(g_tr, z, sizeof z); }
  return e_;
#else
  (void)out; (void)n_words; return cudaErrorNotSupported;
#endif
}

cudaError_t msv_read_profile(unsigned long long out[64], int reset) {
  cudaError_t e = cudaMemcpyFromSymbol(out, g_prof, sizeof(unsigned long long) * 64);
  if (e != cudaSuccess) return e;
#ifdef MSV_PROFILE
  { unsigned long long d[8]; cudaMemcpyFromSymbol(d, g_dbg, sizeof d); out[28] = d[0]; out[29] = d[1]; out[30] = d[2]; out[31] = d[5]; unsigned long long z8[8] = {0}; if (reset) cudaMemcpyToSymbol(g_dbg, z8, sizeof z8); }
  { unsigned long long d[16]; cudaMemcpyFromSymbol(d, g_cnt, sizeof d); for (int k = 0; k < 4; ++k) out[44 + k] = 0; for (int k = 0; k < 16; ++k) if (k < 4) out[44 + k] = d[k]; 
    // [44..47] generic solve / TOI event (calls, cycles); the rest go to [60..63] and the slowest-wait slots that are unused ([58],[59])
    out[58] = d[4]; out[59] = d[5]; out[60] = d[6]; out[61] = d[7]; out[62] = d[8]; out[63] = d[9];
    out[14] = d[10]; out[15] = d[11]; out[42] = d[12]; out[43] = d[13];
    unsigned long long z16[16] = {0}; if (reset) cudaMemcpyToSymbol(g_cnt, z16, sizeof z16);
    unsigned long long sb_[16]; cudaMemcpyFromSymbol(sb_, g_sub, sizeof sb_);
    for (int k = 0; k < 6; ++k) out[20 + k] = sb_[k];     // (slots 16..27 normally hold the slowest group's phases; 20..25 reused when MSV_SUBPROF is read)
    for (int k = 0; k < 8; ++k) out[48 + k] = sb_[8 + k]; // island sub-phases (slots 48.. normally: the slowest group's waits)
    out[26] = sb_[6]; out[27] = sb_[7];                   // longest island_single<NR> / <BC+4> (cycles << 8 | contacts)
    if (reset) cudaMemcpyToSymbol(g_sub, z16, sizeof z16); }
#endif
  if (reset) { unsigned long long z[64] = {0}; e = cudaMemcpyToSymbol(g_prof, z, sizeof z); }
  return e;
}
