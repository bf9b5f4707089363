// msv_env.cuh -- one environment's step, executed by a GROUP of G adjacent
// lanes of a warp (G = agent capacity of the kernel instance): lane g owns
// agent g.  The per-agent phases -- motors, melee rays, broad phase, narrow
// phase, the island of an agent that only touches static bodies, the TOI
// scan, the camera rays -- run on all lanes at once, each on its own agent;
// the cross-agent sequential rules (inventories, deaths, pickups, rewards,
// agent-agent islands, TOI events, contact numbering) run on the group's
// leader lane while the others wait at a group barrier.  The environment's hot
// state (agent sweeps/velocities/fat AABBs, boxes, the touching-contact list)
// lives in one shared-memory column per environment (word w of environment
// slot s at sm[w * T + s]); lanes exchange the pair bit-matrices and small
// results with warp shuffles of width G.
//
// Reference behaviour being reproduced (citations into /root/reference):
//   env  = masurvival/envs/masurvival_env.py   sim = masurvival/simulation.py
//   sem  = masurvival/semantics.py
// and, for the physics, the Box2D v2.3.x routines named at each function.
#pragma once
#include "msv_device.cuh"
#include "msv_types.cuh"
#include "msv_launch.h"

// shared-memory agent fields
enum { F_CX, F_CY, F_A, F_VX, F_VY, F_W, F_C0X, F_C0Y, F_A0, F_ALPHA0, F_SLEEP,
       F_FAT0, F_FAT1, F_FAT2, F_FAT3, F_FLAGS, F_QS, F_QC, F_COUNT };
// shared-memory box fields
enum { G_X, G_Y, G_HX, G_HY, G_AX, G_AY, G_ROT, G_F0, G_F1, G_F2, G_F3, G_COUNT };   // G_F*: fat AABB (b2DynamicTree proxy)
// shared-memory touching-contact fields (a b2Contact with a one-point manifold)
enum { K_META, K_SEQ, K_MTYPE, K_LNX, K_LNY, K_LPX, K_LPY, K_NI, K_TI, K_NM, K_TM, K_COUNT };
// the same words while solve_island() works on a contact (its list entry is dead once the island order is fixed):
// world normal, plane point (static body A) or rA (agent-agent), rB, effective masses
enum { KS_NX = K_SEQ, KS_NY = K_MTYPE, KS_PX = K_LNX, KS_PY = K_LNY, KS_RBX = K_LPX, KS_RBY = K_LPY };

#define FL_ALIVE 1
#define FL_AWAKE 2
#define FL_ISLAND 4
#define FL_MOVED 8

#define KIND_NONE 0
#define KIND_AGENT 1
#define KIND_BOX 2
#define KIND_ITEM 3
#define KIND_HEAL 4
#define KIND_WALL 5

#define STREAM_SHUFFLE 0
#define STREAM_BOX 1
#define STREAM_ZONE 2
#define STREAM_DEATH 3

template <int AC, int BC> struct PairLayout {
  static constexpr int NAA = AC * (AC - 1) / 2;
  static constexpr int NAB = AC * BC;
  static constexpr int P = NAA + NAB + AC * 4;
  static constexpr int PW = (P + 63) / 64;
};

// one touching contact, with its solver scratch (b2ContactVelocityConstraint /
// b2ContactPositionConstraint for a single manifold point)
struct TCon {
  int p, seq;
  int a;     // agent index of body A, or -1 when A is static
  int sid;   // static id of body A (box k, or BC + wall k) when a < 0
  int b;     // agent index of body B
  int flags; // 1 = in island
  Manifold m;
  float ni, ti;
  f2 normal, rA, rB;
  float normalMass, tangentMass;
};

struct BodyS { f2 c; float a; f2 v; float w; float invM, invI; };

// the block's dynamic shared memory (addressed as shared, not through a generic pointer)
extern __shared__ float msv_sm[];


#ifndef MSV_INLINE_MASK
#define MSV_INLINE_MASK 0
#endif
#ifndef MSV_TOI_COOP
#define MSV_TOI_COOP 0   // deal the b2TimeOfImpact calls of SolveTOI out to the group's lanes (0: every lane its own agent's)
#endif
#ifndef MSV_FIXPOINT
#define MSV_FIXPOINT 1   // stop Gauss-Seidel sweeps at a bitwise fixed point (exact); 0 = always run every iteration (development A/B)
#endif
#if (MSV_INLINE_MASK >> 0) & 1
#define COLD0 __device__ __forceinline__
#else
#define COLD0 __device__ __noinline__
#endif
#if (MSV_INLINE_MASK >> 1) & 1
#define COLD1 __device__ __forceinline__
#else
#define COLD1 __device__ __noinline__
#endif
#if (MSV_INLINE_MASK >> 2) & 1
#define COLD2 __device__ __forceinline__
#else
#define COLD2 __device__ __noinline__
#endif
#if (MSV_INLINE_MASK >> 3) & 1
#define COLD3 __device__ __forceinline__
#else
#define COLD3 __device__ __noinline__
#endif
#if (MSV_INLINE_MASK >> 4) & 1
#define COLD4 __device__ __forceinline__
#else
#define COLD4 __device__ __noinline__
#endif

// Counter-based Philox draws of (global env id, episode, step, stream, block): two uniform doubles per block
__device__ __noinline__ double2 philox_uniform2_of(const DevConst& C, uint32_t genv, uint32_t episode, uint32_t step, uint32_t stream, uint32_t blk) {
  uint32_t o[4];
  philox4x32(genv, episode, step, (stream << 16) | blk, C.seed_lo, C.seed_hi, o);
  return make_double2(((double)(o[0] >> 5) * 67108864.0 + (double)(o[1] >> 6)) / 9007199254740992.0,
                      ((double)(o[2] >> 5) * 67108864.0 + (double)(o[3] >> 6)) / 9007199254740992.0);
}

// Everything BaseEnv.reset (env:59-74) takes from the random generator, for episode `episode` of global env
// `genv`, as one record (layout MSV_SP_*): SpawnGrid shuffle (sem:59-79) -> the cells ResetSpawns hands to boxes,
// heals and agents (sem:82-94), RandomizeBoxShapes (sem:97-120), SafeZone centres (sem:739-756).  A pure function
// of (seed, env, episode): k_spare evaluates it ahead of time, the step kernel only when no record is ready.
__device__ __noinline__ void draw_reset(const DevConst& C, uint32_t genv, uint32_t episode, float* rec) {
  const int n = C.grid_n;
  unsigned char perm[64];
  for (int k = 0; k < n; ++k) perm[k] = (unsigned char)k;
  double2 up = make_double2(0.0, 0.0);
  for (int i = n - 1; i >= 1; --i) {
    const uint32_t kd = (uint32_t)(n - 1 - i);
    if (!(kd & 1u)) up = philox_uniform2_of(C, genv, episode, 0u, STREAM_SHUFFLE, kd >> 1);
    const double u = (kd & 1u) ? up.y : up.x;
    const int j = (int)(u * (i + 1));
    const unsigned char t = perm[i]; perm[i] = perm[j]; perm[j] = t;
  }
  int top = n;
  for (int b = 0; b < C.B0; ++b) {
    float hx = C.box_h, hy = C.box_h;
    if (C.box_randomized) {
      double z[2];
      for (int q = 0; q < 2; ++q) {
        const double2 ub = philox_uniform2_of(C, genv, episode, 0u, STREAM_BOX, (uint32_t)(2 * b + q));
        z[q] = sqrt(-2.0 * log(1.0 - ub.x)) * cos(6.283185307179586 * ub.y);
      }
      double w = C.box_avg_w + C.box_std_w * z[0]; if (!(w > C.box_min_w)) w = C.box_min_w;
      double h = C.box_avg_h + C.box_std_h * z[1]; if (!(h > C.box_min_h)) h = C.box_min_h;
      hx = (float)(w / 2.); hy = (float)(h / 2.);
    }
    const int cell = perm[--top];
    rec[MSV_SP_BOX + 4 * b + 0] = C.grid_px[cell]; rec[MSV_SP_BOX + 4 * b + 1] = C.grid_py[cell];
    rec[MSV_SP_BOX + 4 * b + 2] = hx; rec[MSV_SP_BOX + 4 * b + 3] = hy;
  }
  for (int h = 0; h < C.H0; ++h) { const int cell = perm[--top]; rec[MSV_SP_HEAL + 2 * h] = C.grid_px[cell]; rec[MSV_SP_HEAL + 2 * h + 1] = C.grid_py[cell]; }
  for (int i = 0; i < C.A; ++i) { const int cell = perm[--top]; rec[MSV_SP_AGENT + 2 * i] = C.grid_px[cell]; rec[MSV_SP_AGENT + 2 * i + 1] = C.grid_py[cell]; }
  if (C.zone_centers_random) {
    int d = 0;
    for (int z = C.n_zones - 1; z >= 0; --z) {
      const double L = C.floor_size - 2 * C.zone_radiuses[z];
      const double2 uz = philox_uniform2_of(C, genv, episode, 0u, STREAM_ZONE, (uint32_t)(d >> 1)); d += 2;
      rec[MSV_SP_ZONE + 2 * z] = (float)((uz.x * L) - L / 2); rec[MSV_SP_ZONE + 2 * z + 1] = (float)((uz.y * L) - L / 2);
    }
  } else {
    for (int z = 0; z < C.n_zones; ++z) { rec[MSV_SP_ZONE + 2 * z] = (float)C.zone_centers[z][0]; rec[MSV_SP_ZONE + 2 * z + 1] = (float)C.zone_centers[z][1]; }
  }
}

template <int AC, int BC, int HC, int G>
struct Env {
  using PL = PairLayout<AC, BC>;
  static constexpr int P = PL::P, PW = PL::PW, NAA = PL::NAA;
  static constexpr int MAXC = AC <= 4 ? 16 : 24;
  // ---- the leader's scalar state lives in the environment's shared-memory column
  // (L_* words below, accessed through the LI/LF/LU accessors): plain LDS/STS, shared by the
  // out-of-line cold paths without copying, no local-memory mirror.
  enum { L_HEALTH = 0, L_CAUSE = L_HEALTH + AC, L_COOLDOWN = L_CAUSE + AC, L_INV = L_COOLDOWN + AC,
         L_SREW = L_INV + AC, L_SKILLS = L_SREW + AC, L_SEENA = L_SKILLS + AC, L_SEENX = L_SEENA + AC,
         L_KCAUSE = L_SEENX + AC, L_EPRET = L_KCAUSE + AC,
         L_NP = L_EPRET + AC, L_STEPS, L_EPISODE, L_BODYSEQ, L_CONTACTSEQ, L_FIRST, L_OVERFLOW, L_NEWFIX,
         L_ZX, L_ZY, L_ZR, L_ZPHASE, L_ZTCOOL, L_ZTSHRINK, L_ZEND,
         L_STSTEPS, L_STHEALS, L_STBOXES, L_STEPISODES, L_USEHEAL, L_USEBOX, L_NEWBOX,
         L_PREALIVE, L_DMASK, L_NKILLS, L_COUNT };
  static constexpr int SLOTS = AC / G;               // agents per lane
  static constexpr int W_BOX = F_COUNT * AC, W_TC = W_BOX + G_COUNT * BC, W_MISC = W_TC + K_COUNT * MAXC;
  static constexpr int W_ITEM = W_MISC + 2, W_HEAL = W_ITEM + 2 * BC;   // floor item / heal positions (x then y)
  static constexpr int W_LEAD = W_HEAL + 2 * HC;
  static constexpr int W_TOI = W_LEAD + L_COUNT;          // cached TOI per (agent, static body)
  static constexpr int SM_USED = W_TOI + AC * (BC + 4);
  // Shared memory is environment-major: word w of environment slot s sits at msv_sm[s * SM_WORDS + w].
  // SM_WORDS == G (mod 32): the G lanes of a group (same slot, words of G different agents) and the
  // 32/G slots of a warp then fall into 32 different banks, whatever the block size.
  static constexpr int SM_WORDS = SM_USED + ((G - SM_USED % 32) + 32) % 32;
  static constexpr int NR = 3;                       // contacts of a one-agent island kept in registers
  static_assert(AC % G == 0 && G <= 32 && (G & (G - 1)) == 0, "G must be a power of two dividing AC");

  const DevConst& C;
  const DevState& S;
  int es, g, e, N;        // es: my slot in the block (blockDim.x / G slots); g: my lane in the group
  int sb;                 // es * SM_WORDS: base of my environment's shared-memory column
  unsigned gmask;         // the group's lanes within the warp
  bool lead;              // g == 0

  // ---- replicated on every lane of the group (kept equal by share_*())
  int nb, ni, nh;
  unsigned long long ex[PW], tc[PW], en[PW];
  unsigned long long own[PW];   // pairs whose body B is one of this lane's agents
  int ntc;

  __device__ __forceinline__ Env(const DevConst& c, const DevState& s, int es_, int g_, unsigned gmask_, int e_)
      : C(c), S(s), es(es_), g(g_), e(e_), N(c.N), sb(es_ * SM_WORDS), gmask(gmask_), lead(g_ == 0) {
#pragma unroll
    for (int w = 0; w < PW; ++w) own[w] = 0ull;
    for (int i = g; i < AC; i += G) {
      for (int a = 0; a < i; ++a) setb(own, p_aa(a, i));
      for (int k = 0; k < BC; ++k) setb(own, p_ab(i, k));
      for (int k = 0; k < 4; ++k) setb(own, p_aw(i, k));
    }
  }

  // ---- group collectives (width-G shuffles; every lane of the group must call them together)
  DEV void gsync() const { __syncwarp(gmask); }
  template <class V> DEV V bc(V v) const { return __shfl_sync(gmask, v, 0, G); }
  template <class V> DEV V from(V v, int j) const { return __shfl_sync(gmask, v, j, G); }
  DEV unsigned or32(unsigned v) const {
#pragma unroll
    for (int o = 1; o < G; o <<= 1) v |= __shfl_xor_sync(gmask, v, o, G);
    return v;
  }
  DEV unsigned long long or64(unsigned long long v) const {
#pragma unroll
    for (int o = 1; o < G; o <<= 1) v |= __shfl_xor_sync(gmask, v, o, G);
    return v;
  }
  DEV void share_counts() { int c = bc(nb | (ni << 8) | (nh << 16)); nb = c & 255; ni = (c >> 8) & 255; nh = (c >> 16) & 255; }
  DEV void share_bits() {
#pragma unroll
    for (int w = 0; w < PW; ++w) { ex[w] = bc(ex[w]); tc[w] = bc(tc[w]); en[w] = bc(en[w]); }
  }
  // every lane changed only the bits of its own pairs: reassemble the matrices
  DEV void merge_bits() {
#pragma unroll
    for (int w = 0; w < PW; ++w) { ex[w] = or64(ex[w] & own[w]); tc[w] = or64(tc[w] & own[w]); en[w] = or64(en[w] & own[w]); }
  }

  // ---- cold paths.  The functions marked __noinline__ below (rare events and
  // the leader's heavy sequential rules) are compiled once, out of line, and
  // are only ever invoked on a COPY of the environment's registers: the object
  // the hot code works on never has its address taken, so the compiler keeps
  // it in registers instead of spilling every field around the calls.
  DEV void take(const Env& o) {
    nb = o.nb; ni = o.ni; nh = o.nh; ntc = o.ntc;
#pragma unroll
    for (int w = 0; w < PW; ++w) { ex[w] = o.ex[w]; tc[w] = o.tc[w]; en[w] = o.en[w]; }
  }
#define MSV_COLD(call) do { Env c_(*this); c_.call; take(c_); } while (0)
  // MSV_INLINE_MASK (development): bit k set -> the cold functions of class k are inlined into the
  // kernel instead (0 islands, 1 TOI events, 2 contact numbering, 3 deaths/pickups/use-give/box removal, 4 reset)
#ifndef MSV_INLINE_MASK
#define MSV_INLINE_MASK 0
#endif
#define MSV_COLDK(k, call) do { if ((MSV_INLINE_MASK >> (k)) & 1) { call; } else { Env c_(*this); c_.call; take(c_); } } while (0)

  // ---- shared-memory accessors
  DEV float& AG(int f, int i) { return msv_sm[sb + (CHK_IDX(f, F_COUNT) * AC + CHK_IDX(i, AC))]; }
  DEV int& AGF(int i) { return reinterpret_cast<int*>(msv_sm)[sb + (F_FLAGS * AC + CHK_IDX(i, AC))]; }
  DEV float& BX(int f, int k) { return msv_sm[sb + (W_BOX + CHK_IDX(f, G_COUNT) * BC + CHK_IDX(k, BC))]; }
  DEV int& BXROT(int k) { return reinterpret_cast<int*>(msv_sm)[sb + (W_BOX + G_ROT * BC + CHK_IDX(k, BC))]; }
  DEV float& KF(int f, int k) { return msv_sm[sb + (W_TC + CHK_IDX(f, K_COUNT) * MAXC + CHK_IDX(k, MAXC))]; }
  DEV int& KI(int f, int k) { return reinterpret_cast<int*>(msv_sm)[sb + (W_TC + CHK_IDX(f, K_COUNT) * MAXC + CHK_IDX(k, MAXC))]; }
  DEV int& NTC() { return reinterpret_cast<int*>(msv_sm)[sb + (W_MISC + 0)]; }
  DEV float& ITP(int c, int k) { return msv_sm[sb + (W_ITEM + CHK_IDX(c, 2) * BC + CHK_IDX(k, BC))]; }
  DEV float& HLP(int c, int k) { return msv_sm[sb + (W_HEAL + CHK_IDX(c, 2) * HC + CHK_IDX(k, HC))]; }
  DEV int& LI(int k) { return reinterpret_cast<int*>(msv_sm)[sb + (W_LEAD + CHK_IDX(k, L_COUNT))]; }
  DEV unsigned& LU(int k) { return reinterpret_cast<unsigned*>(msv_sm)[sb + (W_LEAD + CHK_IDX(k, L_COUNT))]; }
  DEV float& LF(int k) { return msv_sm[sb + (W_LEAD + CHK_IDX(k, L_COUNT))]; }
  DEV float& TOIA(int i, int k) { return msv_sm[sb + (W_TOI + CHK_IDX(i, AC) * (BC + 4) + CHK_IDX(k, BC + 4))]; }
  DEV int& OVF() { return reinterpret_cast<int*>(msv_sm)[sb + (W_MISC + 1)]; }
  DEV bool alive(int i) { return AGF(i) & FL_ALIVE; }
  DEV bool awake(int i) { return AGF(i) & FL_AWAKE; }
  DEV f2 apos(int i) { return mk2(AG(F_CX, i), AG(F_CY, i)); }
  // K_META: pair | (a + 1) << 8 | sid << 12 | b << 16
  DEV static int meta_pack(int p, int a, int sid, int b) { return p | ((a + 1) << 8) | ((sid < 0 ? 0 : sid) << 12) | (b << 16); }
  DEV static void meta_unpack(int m, int& p, int& a, int& sid, int& b) { p = m & 255; a = ((m >> 8) & 15) - 1; sid = (m >> 12) & 15; b = (m >> 16) & 15; }

  // ---- pair bit helpers
  // (the word index is resolved with an unrolled select so that the matrices stay in registers)
  DEV static bool bit(const unsigned long long* m, int p) {
    unsigned long long w = m[0];
#pragma unroll
    for (int q = 1; q < PW; ++q) if ((p >> 6) == q) w = m[q];
    return (w >> (p & 63)) & 1ull;
  }
  DEV static void setb(unsigned long long* m, int p) {
#pragma unroll
    for (int q = 0; q < PW; ++q) if (PW == 1 || (p >> 6) == q) m[q] |= 1ull << (p & 63);
  }
  DEV static void clrb(unsigned long long* m, int p) {
#pragma unroll
    for (int q = 0; q < PW; ++q) if (PW == 1 || (p >> 6) == q) m[q] &= ~(1ull << (p & 63));
  }
  DEV static int p_aa(int i, int j) { return j * (j - 1) / 2 + i; }  // i < j
  DEV static int p_ab(int i, int k) { return NAA + i * BC + k; }
  DEV static int p_aw(int i, int k) { return NAA + AC * BC + i * 4 + k; }
  // decode pair -> (a, sid, b)
  DEV static void decode(int p, int& a, int& sid, int& b) {
    CHK((unsigned)p < (unsigned)P);
    if (p < NAA) {
      int j = 1; while (j * (j + 1) / 2 <= p) ++j;
      a = p - j * (j - 1) / 2; b = j; sid = -1;
    } else if (p < NAA + AC * BC) {
      int q = p - NAA; a = -1; b = q / BC; sid = q % BC;
    } else {
      int q = p - NAA - AC * BC; a = -1; b = q >> 2; sid = BC + (q & 3);
    }
  }

  // ---- global state I/O -------------------------------------------------
  // Every global load of the environment is issued before the first shared-memory store: the state
  // pointers are generic, so a store to shared memory orders the loads behind it and the load phase
  // would pay the HBM latency once per field group instead of once.
  DEV void load() {
    static_assert(SLOTS == 1, "one agent per lane");
    constexpr int BL = (BC + G - 1) / G, HL = (HC + G - 1) / G;   // boxes / heals per lane
    const int i = g;
    const bool mine = i < C.A;
    float4 k0 = make_float4(0.f, 0.f, 0.f, 0.f), k1 = k0, ft = k0;
    if (mine) { k0 = S.akin0[i * N + e]; k1 = S.akin1[i * N + e]; ft = S.afat[i * N + e]; }
    float4 b0[BL], it0[BL]; int4 b1[BL]; float2 hl[HL];
#pragma unroll
    for (int q = 0; q < BL; ++q) {               // slots past the list lengths hold stale data that is never read
      const int k = g + q * G;
      if (k < BC) { b0[q] = S.box0[k * N + e]; b1[q] = S.box1[k * N + e]; it0[q] = S.item0[k * N + e]; }
    }
#pragma unroll
    for (int q = 0; q < HL; ++q) { const int k = g + q * G; if (k < HC) hl[q] = S.heal[k * N + e]; }
    int4 ai[AC]; float srw[AC], epr[AC]; int skl[AC];
    int4 h0 = make_int4(0, 0, 0, 0), h1 = h0, zi = h0, sm_ = h0; float4 zc = make_float4(0.f, 0.f, 0.f, 0.f);
    unsigned long long lx[PW], lt[PW], ln[PW];
    if (lead) {
#pragma unroll
      for (int j = 0; j < AC; ++j) {
        ai[j] = j < C.A ? S.aint[j * N + e] : make_int4(0, MSV_CAUSE_NONE, 0, 0);
        srw[j] = S.sreward[j * N + e]; skl[j] = S.skills[j * N + e]; epr[j] = S.epret[j * N + e];
      }
      h0 = S.hdr0[e]; h1 = S.hdr1[e];
#pragma unroll
      for (int w = 0; w < PW; ++w) { lx[w] = S.pex[w * N + e]; lt[w] = S.ptc[w * N + e]; ln[w] = S.pen[w * N + e]; }
      zc = S.zonecur[e]; zi = S.zoneint[e]; sm_ = S.smisc[e];
    }
    // ---- shared-memory stores
    if (mine) {
      AG(F_CX, i) = k0.x; AG(F_CY, i) = k0.y; AG(F_A, i) = k0.z; AG(F_VX, i) = k0.w;
      AG(F_VY, i) = k1.x; AG(F_W, i) = k1.y; AG(F_SLEEP, i) = k1.z; AGF(i) = __float_as_int(k1.w) & 3;
      AG(F_FAT0, i) = ft.x; AG(F_FAT1, i) = ft.y; AG(F_FAT2, i) = ft.z; AG(F_FAT3, i) = ft.w;
      AG(F_C0X, i) = k0.x; AG(F_C0Y, i) = k0.y; AG(F_A0, i) = k0.z; AG(F_ALPHA0, i) = 0.0f;
      AG(F_QS, i) = 0.0f; AG(F_QC, i) = 1.0f;
    } else AGF(i) = 0;
#pragma unroll
    for (int q = 0; q < BL; ++q) {
      const int k = g + q * G;
      if (k < BC) { put_box(k, b0[q], b1[q]); ITP(0, k) = it0[q].x; ITP(1, k) = it0[q].y; }
    }
#pragma unroll
    for (int q = 0; q < HL; ++q) { const int k = g + q * G; if (k < HC) { HLP(0, k) = hl[q].x; HLP(1, k) = hl[q].y; } }
    nb = ni = nh = 0;
#pragma unroll
    for (int w = 0; w < PW; ++w) { ex[w] = 0ull; tc[w] = 0ull; en[w] = 0ull; }
    if (lead) {
#pragma unroll
      for (int j = 0; j < AC; ++j) {
        LI(L_HEALTH + (j)) = ai[j].x; LI(L_CAUSE + (j)) = ai[j].y; LI(L_COOLDOWN + (j)) = ai[j].z; LI(L_INV + (j)) = ai[j].w;
        LF(L_SREW + (j)) = srw[j]; LI(L_SKILLS + (j)) = skl[j]; LF(L_EPRET + (j)) = epr[j];
      }
      nb = h0.x & 255; ni = (h0.x >> 8) & 255; nh = (h0.x >> 16) & 255; LI(L_NP) = (h0.x >> 24) & 255;
      LI(L_STEPS) = h0.y; LI(L_EPISODE) = h0.z; LI(L_BODYSEQ) = h0.w;
      LI(L_CONTACTSEQ) = h1.x; LI(L_FIRST) = h1.y; LI(L_OVERFLOW) = h1.z; LI(L_NEWFIX) = h1.w;
#pragma unroll
      for (int w = 0; w < PW; ++w) { ex[w] = lx[w]; tc[w] = lt[w]; en[w] = ln[w]; }
      LF(L_ZX) = zc.x; LF(L_ZY) = zc.y; LF(L_ZR) = zc.z; LI(L_ZPHASE) = zi.x; LI(L_ZTCOOL) = zi.y; LI(L_ZTSHRINK) = zi.z; LI(L_ZEND) = zi.w;
      LI(L_STSTEPS) = sm_.x; LI(L_STHEALS) = sm_.y; LI(L_STBOXES) = sm_.z; LI(L_STEPISODES) = sm_.w;
      NTC() = 0; OVF() = 0;
    }
    ntc = 0;
    gsync();
    share_counts(); share_bits();
  }
  // shared-memory record of a box (shape expanded, fat AABB computed once per box and step instead of once per pair test)
  DEV void put_box(int dst, float4 b0, int4 b1) {
    BX(G_X, dst) = b0.x; BX(G_Y, dst) = b0.y;
    SBox t; sb_set_shape(t, b0.z, b0.w, (b1.y >> 1) & 1);
    BX(G_HX, dst) = t.hx; BX(G_HY, dst) = t.hy; BX(G_AX, dst) = t.ax; BX(G_AY, dst) = t.ay; BXROT(dst) = t.rot;
    t.px = b0.x; t.py = b0.y; t.qs = 0.0f; t.qc = 1.0f; t.ang = 0.0f;
    float ft[4]; sb_fat(t, ft);
    BX(G_F0, dst) = ft[0]; BX(G_F1, dst) = ft[1]; BX(G_F2, dst) = ft[2]; BX(G_F3, dst) = ft[3];
  }
  // read box at global slot `src` into shared slot `dst`
  DEV void load_box(int dst, int src) { put_box(dst, S.box0[src * N + e], S.box1[src * N + e]); }
  DEV void store() {
    gsync();
    for (int i = g; i < C.A; i += G) {
      S.akin0[i * N + e] = make_float4(AG(F_CX, i), AG(F_CY, i), AG(F_A, i), AG(F_VX, i));
      S.akin1[i * N + e] = make_float4(AG(F_VY, i), AG(F_W, i), AG(F_SLEEP, i), __int_as_float(AGF(i) & 3));
      S.afat[i * N + e] = make_float4(AG(F_FAT0, i), AG(F_FAT1, i), AG(F_FAT2, i), AG(F_FAT3, i));
    }
    if (lead) {
#pragma unroll
      for (int i = 0; i < AC; ++i) {
        if (i < C.A) S.aint[i * N + e] = make_int4(LI(L_HEALTH + (i)), LI(L_CAUSE + (i)), LI(L_COOLDOWN + (i)), LI(L_INV + (i)));
        S.sreward[i * N + e] = LF(L_SREW + (i)); S.skills[i * N + e] = LI(L_SKILLS + (i));
        S.epret[i * N + e] = LF(L_EPRET + (i));
      }
      S.hdr0[e] = make_int4(nb | (ni << 8) | (nh << 16) | (LI(L_NP) << 24), LI(L_STEPS), LI(L_EPISODE), LI(L_BODYSEQ));
      S.hdr1[e] = make_int4(LI(L_CONTACTSEQ), LI(L_FIRST), LI(L_OVERFLOW) + OVF(), LI(L_NEWFIX));
      // box positions/shapes only change on spawn/despawn, which write through
#pragma unroll
      for (int w = 0; w < PW; ++w) { S.pex[w * N + e] = ex[w]; S.ptc[w * N + e] = tc[w]; S.pen[w * N + e] = en[w]; }
      S.zonecur[e] = make_float4(LF(L_ZX), LF(L_ZY), LF(L_ZR), 0.0f);
      S.zoneint[e] = make_int4(LI(L_ZPHASE), LI(L_ZTCOOL), LI(L_ZTSHRINK), LI(L_ZEND));
      S.smisc[e] = make_int4(LI(L_STSTEPS), LI(L_STHEALS), LI(L_STBOXES), LI(L_STEPISODES));
    }
  }

  // ---- geometry helpers ---------------------------------------------------
  DEV SBox static_box(int sid) {
    SBox b;
    if (sid < BC) {
      b.px = BX(G_X, sid); b.py = BX(G_Y, sid); b.qs = 0.0f; b.qc = 1.0f; b.ang = 0.0f;
      b.hx = BX(G_HX, sid); b.hy = BX(G_HY, sid); b.ax = BX(G_AX, sid); b.ay = BX(G_AY, sid); b.rot = BXROT(sid);
    } else {
      const WallC& w = C.walls[sid - BC];
      b.px = w.px; b.py = w.py; b.qs = w.qs; b.qc = w.qc; b.ang = w.ang;
      b.hx = C.wall_hx; b.hy = C.wall_hy; b.ax = 1.0f; b.ay = 1.0f; b.rot = 0;
    }
    return b;
  }
  DEV void static_fat(int sid, float out[4]) {
    if (sid < BC) { out[0] = BX(G_F0, sid); out[1] = BX(G_F1, sid); out[2] = BX(G_F2, sid); out[3] = BX(G_F3, sid); }
    else { const WallC& w = C.walls[sid - BC]; out[0] = w.fat[0]; out[1] = w.fat[1]; out[2] = w.fat[2]; out[3] = w.fat[3]; }
  }
  DEV void agent_fat(int i, float out[4]) {
    out[0] = AG(F_FAT0, i); out[1] = AG(F_FAT1, i); out[2] = AG(F_FAT2, i); out[3] = AG(F_FAT3, i);
  }
  DEV int static_seq(int sid) { return sid < BC ? S.boxseq[sid * N + e] : C.B0 + C.H0 + (sid - BC); }
  DEV int agent_seq(int i) { return C.B0 + C.H0 + 4 + i; }
  DEV void wake(int i) {  // b2Body::SetAwake(true)
    int f = AGF(i);
    if (!(f & FL_AWAKE)) { AGF(i) = f | FL_AWAKE; AG(F_SLEEP, i) = 0.0f; }
  }
  DEV void wake_all(unsigned m) { for (int i = 0; i < C.A; ++i) if ((m >> i) & 1u) wake(i); }
  DEV void sleep_body(int i) {  // b2Body::SetAwake(false)
    AGF(i) &= ~FL_AWAKE; AG(F_SLEEP, i) = 0.0f; AG(F_VX, i) = 0.0f; AG(F_VY, i) = 0.0f; AG(F_W, i) = 0.0f;
  }
  DEV int team_of(int i) { return i < C.A / 2 ? 0 : 1; }  // sem:957-966

  // closest hit of the segment p1->p2 over every fixture except agent `self`
  // (whose own circle contains p1 and therefore always misses); minimum
  // fraction over independent b2Shape::RayCast tests (sim:431-439, 471-484).
  // Every exact test is preceded by a conservative reject (segment AABB vs a
  // bound of the shape): it can only skip shapes the exact test would miss.
  DEV int raycast(f2 p1, f2 p2, int self, int& idx, float& frac) {
    int kind = KIND_NONE; idx = -1; frac = 0.0f; float f;
    const float lx = fmin_(p1.x, p2.x), ly = fmin_(p1.y, p2.y), ux = fmax_(p1.x, p2.x), uy = fmax_(p1.y, p2.y);
    auto far_from = [&](float cx, float cy, float rad) {  // rad already includes slack
      return cx + rad < lx || cx - rad > ux || cy + rad < ly || cy - rad > uy;
    };
    for (int k = 0; k < nb; ++k) {
      float bxr = BX(G_HX, k) + BX(G_HY, k) + 0.01f;     // |hx|+|hy| >= circumradius
      if (far_from(BX(G_X, k), BX(G_Y, k), bxr)) continue;
      if (ray_box(static_box(k), p1, p2, f) && (kind == KIND_NONE || f < frac)) { kind = KIND_BOX; idx = k; frac = f; }
    }
    for (int k = 0; k < ni; ++k) {
      const float itx = ITP(0, k), ity = ITP(1, k);
      if (far_from(itx, ity, C.item_r + 0.01f)) continue;
      if (ray_circle(mk2(itx, ity), C.item_r, p1, p2, f) && (kind == KIND_NONE || f < frac)) { kind = KIND_ITEM; idx = k; frac = f; }
    }
    for (int k = 0; k < nh; ++k) {
      const float hx_ = HLP(0, k), hy_ = HLP(1, k);
      if (far_from(hx_, hy_, C.heal_r + 0.01f)) continue;
      if (ray_circle(mk2(hx_, hy_), C.heal_r, p1, p2, f) && (kind == KIND_NONE || f < frac)) { kind = KIND_HEAL; idx = k; frac = f; }
    }
    for (int k = 0; k < 4; ++k) {
      const WallC& w = C.walls[k];                        // fat AABB = tight AABB + 0.11
      if (w.fat[2] < lx || w.fat[0] > ux || w.fat[3] < ly || w.fat[1] > uy) continue;
      if (ray_box(static_box(BC + k), p1, p2, f) && (kind == KIND_NONE || f < frac)) { kind = KIND_WALL; idx = k; frac = f; }
    }
    for (int j = 0; j < C.A; ++j) {
      if (j == self || !alive(j)) continue;
      if (far_from(AG(F_CX, j), AG(F_CY, j), C.agent_r + 0.01f)) continue;
      if (ray_circle(apos(j), C.agent_r, p1, p2, f) && (kind == KIND_NONE || f < frac)) { kind = KIND_AGENT; idx = j; frac = f; }
    }
    return kind;
  }

  // Health._change_health (sem:490-500)                                [leader]
  DEV void agent_change_health(int i, int delta, int cz) {
    if (!alive(i)) return;
    if (C.teams && cz == MSV_CAUSE_TEAM0 + team_of(i)) return;  // immunities sem:942-946
    LI(L_HEALTH + i) += delta; LI(L_CAUSE + i) = cz;
  }
  DEV void box_change_health(int k, int delta, int cz) {
    int4 b1 = S.box1[k * N + e];
    if (!(b1.y & 1)) return;                                      // Q9 sem:491-492
    if (b1.w != MSV_CAUSE_NONE && cz != b1.w) return;             // sem:497-498
    b1.x += delta; b1.z = cz;
    S.box1[k * N + e] = b1;
  }
  DEV int inv_n(int i) { return LI(L_INV + (i)) & 7; }
  DEV int inv_kind(int i, int s) { return (LI(L_INV + (i)) >> (4 + 2 * s)) & 3; }
  DEV void inv_push(int i, int kind, float4 payload) {
    int n = inv_n(i);
    LI(L_INV + (i)) = (LI(L_INV + (i)) & ~(3 << (4 + 2 * n)) & ~7) | (kind << (4 + 2 * n)) | (n + 1);
    if (kind == MSV_ITEM_BOX) S.ainv[(i * 4 + n) * N + e] = payload;
  }
  DEV int inv_pop(int i, float4& payload) {  // list.pop(-1)
    int n = inv_n(i) - 1;
    int kind = inv_kind(i, n);
    if (kind == MSV_ITEM_BOX) payload = S.ainv[(i * 4 + n) * N + e];
    LI(L_INV + (i)) = (LI(L_INV + (i)) & ~7) | n;
    return kind;
  }

  // ---- list maintenance (stable compaction, sim:185-189)            [leader]
  // shift the AB pair column k+1.. down by one for every agent
  COLD3 void remove_box(int k) {
    for (int i = 0; i < C.A; ++i) {   // b2World::DestroyBody -> contacts die, touching ones wake
      int p = p_ab(i, k);
      if (bit(ex, p) && bit(tc, p)) wake(i);
      for (int q = k; q + 1 < nb; ++q) {
        int pd = p_ab(i, q), ps = p_ab(i, q + 1);
        if (bit(ex, ps)) { setb(ex, pd); S.pseq[pd * N + e] = S.pseq[ps * N + e]; S.pimp[pd * N + e] = S.pimp[ps * N + e]; } else clrb(ex, pd);
        if (bit(tc, ps)) setb(tc, pd); else clrb(tc, pd);
        if (bit(en, ps)) setb(en, pd); else clrb(en, pd);
      }
      int pl = p_ab(i, nb - 1);
      clrb(ex, pl); clrb(tc, pl); clrb(en, pl);
    }
    for (int q = k; q + 1 < nb; ++q) {
      S.box0[q * N + e] = S.box0[(q + 1) * N + e];
      S.box1[q * N + e] = S.box1[(q + 1) * N + e];
      S.boxseq[q * N + e] = S.boxseq[(q + 1) * N + e];
      BX(G_X, q) = BX(G_X, q + 1); BX(G_Y, q) = BX(G_Y, q + 1); BX(G_HX, q) = BX(G_HX, q + 1);
      BX(G_HY, q) = BX(G_HY, q + 1); BX(G_AX, q) = BX(G_AX, q + 1); BX(G_AY, q) = BX(G_AY, q + 1);
      BXROT(q) = BXROT(q + 1);
      BX(G_F0, q) = BX(G_F0, q + 1); BX(G_F1, q) = BX(G_F1, q + 1); BX(G_F2, q) = BX(G_F2, q + 1); BX(G_F3, q) = BX(G_F3, q + 1);
    }
    nb--;
  }
  DEV void remove_item(int k) {
    for (int q = k; q + 1 < ni; ++q) { S.item0[q * N + e] = S.item0[(q + 1) * N + e]; S.item1[q * N + e] = S.item1[(q + 1) * N + e]; ITP(0, q) = ITP(0, q + 1); ITP(1, q) = ITP(1, q + 1); }
    ni--;
  }
  DEV void remove_heal(int k) {
    for (int q = k; q + 1 < nh; ++q) { S.heal[q * N + e] = S.heal[(q + 1) * N + e]; S.healseq[q * N + e] = S.healseq[(q + 1) * N + e]; HLP(0, q) = HLP(0, q + 1); HLP(1, q) = HLP(1, q + 1); }
    nh--;
  }
  DEV void add_item(float x, float y, float hx, float hy, int owner) {  // Item.drop sem:143-148
    if (ni >= BC) { LI(L_OVERFLOW)++; return; }
    S.item0[ni * N + e] = make_float4(x, y, hx, hy); ITP(0, ni) = x; ITP(1, ni) = y;
    S.item1[ni * N + e] = make_int2(owner, LI(L_BODYSEQ)++);
    ni++;
  }
  DEV void add_heal(float x, float y) {
    if (nh >= HC) { LI(L_OVERFLOW)++; return; }
    S.heal[nh * N + e] = make_float2(x, y); HLP(0, nh) = x; HLP(1, nh) = y;
    S.healseq[nh * N + e] = LI(L_BODYSEQ)++;
    nh++;
  }
  DEV void kill_agent(int i) {  // b2World::DestroyBody for an agent
    for (int j = 0; j < C.A; ++j) {
      if (j == i) continue;
      int p = i < j ? p_aa(i, j) : p_aa(j, i);
      if (bit(ex, p) && bit(tc, p)) wake(j);
      clrb(ex, p); clrb(tc, p); clrb(en, p);
    }
    for (int k = 0; k < BC + 4; ++k) {
      int p = k < BC ? p_ab(i, k) : p_aw(i, k - BC);
      clrb(ex, p); clrb(tc, p); clrb(en, p);
    }
    AGF(i) = 0;
  }

  // ======================================================================
  //                               PHYSICS
  // ======================================================================
  // b2ContactManager::FindNewContacts + AddPair over every body pair whose
  // fat AABBs overlap and that has no contact yet; new contacts are numbered
  // in ascending (proxyIdA, proxyIdB) order (creation sequence surrogate).
  // candidate pairs whose body B is agent j
  // only_moved: b2BroadPhase::UpdatePairs queries the proxies that moved in this solve; a pair
  // neither of whose proxies moved cannot have started to overlap
  DEV void candidates_of(int j, unsigned long long* cand, bool only_moved = false) {
    const int fj_ = AGF(j);
    if (!(fj_ & FL_ALIVE)) return;
    const bool mj = !only_moved || (fj_ & FL_MOVED);
    float fj[4]; agent_fat(j, fj);
    for (int i = 0; i < j; ++i) {
      const int fi_ = AGF(i);
      if (!(fi_ & FL_ALIVE)) continue;
      if (!mj && !(fi_ & FL_MOVED)) continue;
      int p = p_aa(i, j);
      if (bit(ex, p)) continue;
      float fi[4]; agent_fat(i, fi);
      if (aabb_overlap(fi, fj)) setb(cand, p);
    }
    if (!mj) return;
    for (int k = 0; k < BC + 4; ++k) {
      if (k < BC && k >= nb) continue;
      int p = k < BC ? p_ab(j, k) : p_aw(j, k - BC);
      if (bit(ex, p)) continue;
      float fs[4]; static_fat(k, fs);
      if (aabb_overlap(fj, fs)) setb(cand, p);
    }
  }
  // [leader] create the candidate contacts in proxy-pair order
  COLD2 void number_candidates(unsigned long long* cand) {
    for (;;) {
      int best = -1; unsigned bestKey = 0xFFFFFFFFu;
      for (int w = 0; w < PW; ++w) {
        unsigned long long m = cand[w];
        while (m) {
          int p = w * 64 + __ffsll((long long)m) - 1; m &= m - 1;
          int a, sid, b; decode(p, a, sid, b);
          int s1 = a >= 0 ? agent_seq(a) : static_seq(sid), s2 = agent_seq(b);
          int lo = s1 < s2 ? s1 : s2, hi = s1 < s2 ? s2 : s1;
          unsigned key = ((unsigned)lo << 16) | (unsigned)hi;
          if (key < bestKey) { bestKey = key; best = p; }
        }
      }
      if (best < 0) break;
      clrb(cand, best);
      setb(ex, best); setb(en, best); clrb(tc, best);
      S.pseq[best * N + e] = (uint32_t)(++LI(L_CONTACTSEQ));
      S.pimp[best * N + e] = make_float2(0.0f, 0.0f);
    }
  }
  // [all lanes] every lane tests the pairs of its own agents; the leader numbers the new contacts
  DEV void find_new_contacts(bool only_moved = false) {
    unsigned long long cand[PW];
#pragma unroll
    for (int w = 0; w < PW; ++w) cand[w] = 0ull;
    for (int j = g; j < C.A; j += G) candidates_of(j, cand, only_moved);
    bool any = false;
#pragma unroll
    for (int w = 0; w < PW; ++w) { cand[w] = or64(cand[w]); any |= cand[w] != 0ull; }
    if (any) {                               // group-uniform
      if (lead) {
        int nset = 0;
#pragma unroll
        for (int w = 0; w < PW; ++w) nset += __popcll(cand[w]);
        if (nset == 1) {                       // one new contact (the usual case): no ordering to do
          int p = 0;
#pragma unroll
          for (int w = 0; w < PW; ++w) if (cand[w]) p = w * 64 + __ffsll((long long)cand[w]) - 1;
          setb(ex, p); setb(en, p); clrb(tc, p);
          S.pseq[p * N + e] = (uint32_t)(++LI(L_CONTACTSEQ));
          S.pimp[p * N + e] = make_float2(0.0f, 0.0f);
        } else { RARE_BEGIN(); unsigned long long cc[PW]; for (int w = 0; w < PW; ++w) cc[w] = cand[w]; MSV_COLDK(2, number_candidates(cc)); RARE_END(6); }
      }
      share_bits();
    }
  }
  // [leader] the same inside a TOI event: only agent b's proxy moved (b2BroadPhase::UpdatePairs queries the
  // moved proxies), so only pairs with b can have started to overlap
  DEV void find_new_contacts_of(int b) {
    unsigned long long cand[PW];
#pragma unroll
    for (int w = 0; w < PW; ++w) cand[w] = 0ull;
    candidates_of(b, cand);                      // (i < b, b) and b against the static bodies
    float fb[4]; agent_fat(b, fb);
    for (int j = b + 1; j < C.A; ++j) {          // (b, j > b)
      if (!(AGF(j) & FL_ALIVE)) continue;
      const int p = p_aa(b, j);
      if (bit(ex, p)) continue;
      float fj[4]; agent_fat(j, fj);
      if (aabb_overlap(fb, fj)) setb(cand, p);
    }
    bool any = false;
#pragma unroll
    for (int w = 0; w < PW; ++w) any |= cand[w] != 0ull;
    if (any) number_candidates(cand);
  }

  // evaluate the manifold of pair (a|sid, b) at the bodies' current transforms
  DEV bool evaluate(int a, int sid, int b, Manifold& m) {
    if (a >= 0) return collide_circles(apos(a), apos(b), C.agent_r, C.agent_r, m);
    return collide_box_circle(static_box(sid), apos(b), C.agent_r, m);
  }

  // append a touching contact to the environment's shared list (any lane)
  DEV void tcon_add(int p, int a, int sid, int b, const Manifold& m, float nimp, float timp) {
    CHK((unsigned)p < (unsigned)P && (unsigned)b < (unsigned)AC && a < AC && sid < BC + 4);
    int k = atomicAdd(&NTC(), 1);
    if (k >= MAXC) { atomicAdd(&OVF(), 1); return; }
    KI(K_META, k) = meta_pack(p, a, sid, b); KI(K_SEQ, k) = (int)S.pseq[p * N + e];
    KI(K_MTYPE, k) = m.type; KF(K_LNX, k) = m.localNormal.x; KF(K_LNY, k) = m.localNormal.y;
    KF(K_LPX, k) = m.localPoint.x; KF(K_LPY, k) = m.localPoint.y; KF(K_NI, k) = nimp; KF(K_TI, k) = timp;
  }

  // b2Contact::Update for one pair; returns touching.  Bodies to wake are
  // collected in `wakem` (the caller applies them); appends to the list.
  DEV bool contact_update(int p, int a, int sid, int b, bool list, unsigned& wakem, Manifold* mout = nullptr) {
    Manifold m; bool touching = evaluate(a, sid, b, m);
    if (mout) *mout = m;
    bool was = bit(tc, p);
    setb(en, p);
    float2 imp = make_float2(0.0f, 0.0f);
    if (touching && was) imp = S.pimp[p * N + e];
    else if (was || touching) S.pimp[p * N + e] = imp;
    if (touching != was) { if (a >= 0) wakem |= 1u << a; wakem |= 1u << b; }
    if (touching) setb(tc, p); else clrb(tc, p);
    if (touching && list) tcon_add(p, a, sid, b, m, imp.x, imp.y);
    return touching;
  }

  // b2ContactManager::Collide.  Every lane updates the contacts whose body B
  // is one of its agents.  SetAwake calls are applied after the pass: a contact
  // between two sleeping bodies is skipped by Box2D, and re-evaluating it for
  // unmoved bodies returns the state it already has.
  __device__ __forceinline__ void collide() {
    if (lead) NTC() = 0;
    gsync();
    unsigned wakem = 0;
#pragma unroll
    for (int w = 0; w < PW; ++w) {
      unsigned long long mbits = ex[w] & own[w];
      while (mbits) {
        int p = w * 64 + __ffsll((long long)mbits) - 1; mbits &= mbits - 1;
        int a, sid, b; decode(p, a, sid, b);
        bool activeA = a >= 0 && awake(a), activeB = awake(b);
        if (!activeA && !activeB) {
          // both asleep/static: Box2D keeps the stale manifold; it is only ever
          // used if the island DFS wakes one of them -> evaluate it lazily now
          if (bit(tc, p)) { Manifold m; if (evaluate(a, sid, b, m)) { float2 imp = S.pimp[p * N + e]; tcon_add(p, a, sid, b, m, imp.x, imp.y); } }
          continue;
        }
        float fa[4], fb[4];
        if (a >= 0) agent_fat(a, fa); else static_fat(sid, fa);
        agent_fat(b, fb);
        if (!aabb_overlap(fa, fb)) {  // b2ContactManager::Destroy
          if (bit(tc, p)) { if (a >= 0) wakem |= 1u << a; wakem |= 1u << b; }
          clrb(ex, p); clrb(tc, p); clrb(en, p);
          continue;
        }
        contact_update(p, a, sid, b, true, wakem);
      }
    }
    merge_bits();
    wakem = or32(wakem);
    gsync();                                 // every lane has read the awake flags
    for (int i = g; i < C.A; i += G) if ((wakem >> i) & 1u) wake(i);
    gsync();
    ntc = NTC(); if (ntc > MAXC) ntc = MAXC;
  }

  // ---- contact solver (single manifold point) ----------------------------
  DEV BodyS body_of(int a, int sid) {
    BodyS s;
    if (a >= 0) {
      s.c = apos(a); s.a = AG(F_A, a); s.v = mk2(AG(F_VX, a), AG(F_VY, a)); s.w = AG(F_W, a);
      s.invM = C.inv_mass; s.invI = C.inv_I;
    } else {
      SBox bx = static_box(sid);
      s.c = mk2(bx.px, bx.py); s.a = bx.ang; s.v = mk2(0.0f, 0.0f); s.w = 0.0f; s.invM = 0.0f; s.invI = 0.0f;
    }
    return s;
  }
  DEV void put_vel(int a, const BodyS& s) { if (a >= 0) { AG(F_VX, a) = s.v.x; AG(F_VY, a) = s.v.y; AG(F_W, a) = s.w; } }
  DEV void put_pos(int a, const BodyS& s) { if (a >= 0) { AG(F_CX, a) = s.c.x; AG(F_CY, a) = s.c.y; AG(F_A, a) = s.a; } }

  // b2ContactSolver::InitializeVelocityConstraints + b2WorldManifold::Initialize
  DEV void init_velocity(TCon& t) {
    BodyS A = body_of(t.a, t.sid), B = body_of(t.b, -1);
    f2 normal, point;
    if (t.m.type == 0) {
      normal = mk2(1.0f, 0.0f);
      f2 pointA = A.c, pointB = B.c;
      if (vlen2(vsub(pointA, pointB)) > B2_EPS * B2_EPS) { normal = vsub(pointB, pointA); vnormalize(normal); }
      f2 pA = vadd(pointA, vmul(C.agent_r, normal));
      f2 pB = vsub(pointB, vmul(C.agent_r, normal));
      point = vmul(0.5f, vadd(pA, pB));
    } else {
      SBox bx = static_box(t.sid);
      normal = qmul(bx.qs, bx.qc, t.m.localNormal);
      f2 planePoint = sb_mul(bx, t.m.localPoint);
      f2 clipPoint = B.c;
      f2 pA = vadd(clipPoint, vmul(B2_POLY_RADIUS - vdot(vsub(clipPoint, planePoint), normal), normal));
      f2 pB = vsub(clipPoint, vmul(C.agent_r, normal));
      point = vmul(0.5f, vadd(pA, pB));
    }
    t.normal = normal;
    t.rA = vsub(point, A.c); t.rB = vsub(point, B.c);
    float rnA = vcross(t.rA, normal), rnB = vcross(t.rB, normal);
    float kNormal = A.invM + B.invM + A.invI * rnA * rnA + B.invI * rnB * rnB;
    t.normalMass = kNormal > 0.0f ? 1.0f / kNormal : 0.0f;
    f2 tangent = cross_vs(normal, 1.0f);
    float rtA = vcross(t.rA, tangent), rtB = vcross(t.rB, tangent);
    float kTangent = A.invM + B.invM + A.invI * rtA * rtA + B.invI * rtB * rtB;
    t.tangentMass = kTangent > 0.0f ? 1.0f / kTangent : 0.0f;
    // restitution 0: velocityBias stays 0
  }
  DEV void apply_impulse(BodyS& A, BodyS& B, const TCon& t, f2 Pv) {
    A.v = vsub(A.v, vmul(A.invM, Pv)); A.w -= A.invI * vcross(t.rA, Pv);
    B.v = vadd(B.v, vmul(B.invM, Pv)); B.w += B.invI * vcross(t.rB, Pv);
  }
  DEV void warm_start(TCon& t) {
    BodyS A = body_of(t.a, t.sid), B = body_of(t.b, -1);
    f2 tangent = cross_vs(t.normal, 1.0f);
    f2 Pv = vadd(vmul(t.ni, t.normal), vmul(t.ti, tangent));
    A.w -= A.invI * vcross(t.rA, Pv); A.v = vsub(A.v, vmul(A.invM, Pv));
    B.w += B.invI * vcross(t.rB, Pv); B.v = vadd(B.v, vmul(B.invM, Pv));
    put_vel(t.a, A); put_vel(t.b, B);
  }
  // b2ContactSolver::SolveVelocityConstraints, one contact
  DEV void solve_velocity(TCon& t) {
    BodyS A = body_of(t.a, t.sid), B = body_of(t.b, -1);
    f2 normal = t.normal, tangent = cross_vs(normal, 1.0f);
    {
      f2 dv = vsub(vsub(vadd(B.v, cross_sv(B.w, t.rB)), A.v), cross_sv(A.w, t.rA));
      float vt = vdot(dv, tangent) - 0.0f;
      float lambda = t.tangentMass * (-vt);
      float maxFriction = C.friction * t.ni;
      float newImpulse = fclamp_(t.ti + lambda, -maxFriction, maxFriction);
      lambda = newImpulse - t.ti; t.ti = newImpulse;
      apply_impulse(A, B, t, vmul(lambda, tangent));
    }
    {
      f2 dv = vsub(vsub(vadd(B.v, cross_sv(B.w, t.rB)), A.v), cross_sv(A.w, t.rA));
      float vn = vdot(dv, normal);
      float lambda = -t.normalMass * (vn - 0.0f);
      float newImpulse = fmax_(t.ni + lambda, 0.0f);
      lambda = newImpulse - t.ni; t.ni = newImpulse;
      apply_impulse(A, B, t, vmul(lambda, normal));
    }
    put_vel(t.a, A); put_vel(t.b, B);
  }
  // b2ContactSolver::SolvePositionConstraints / SolveTOIPositionConstraints, one contact
  DEV float solve_position(const TCon& t, bool toi, int toiAgent) {
    BodyS A = body_of(t.a, t.sid), B = body_of(t.b, -1);
    float mA = A.invM, iA = A.invI, mB = B.invM, iB = B.invI;
    if (toi) {  // only the two TOI bodies move; the static one has no mass anyway
      if (t.a != toiAgent) { mA = 0.0f; iA = 0.0f; }
      if (t.b != toiAgent) { mB = 0.0f; iB = 0.0f; }
    }
    f2 normal, point; float separation;
    if (t.m.type == 0) {
      normal = vsub(B.c, A.c); vnormalize(normal);
      point = vmul(0.5f, vadd(A.c, B.c));
      separation = vdot(vsub(B.c, A.c), normal) - C.agent_r - C.agent_r;
    } else {
      SBox bx = static_box(t.sid);
      normal = qmul(bx.qs, bx.qc, t.m.localNormal);
      f2 planePoint = sb_mul(bx, t.m.localPoint);
      separation = vdot(vsub(B.c, planePoint), normal) - B2_POLY_RADIUS - C.agent_r;
      point = B.c;
    }
    f2 rA = vsub(point, A.c), rB = vsub(point, B.c);
    float Cc = fclamp_((toi ? B2_TOI_BAUMGARTE : B2_BAUMGARTE) * (separation + B2_LINEAR_SLOP), -B2_MAX_LIN_CORR, 0.0f);
    float rnA = vcross(rA, normal), rnB = vcross(rB, normal);
    float K = mA + mB + iA * rnA * rnA + iB * rnB * rnB;
    float impulse = K > 0.0f ? -Cc / K : 0.0f;
    f2 Pv = vmul(impulse, normal);
    A.c = vsub(A.c, vmul(mA, Pv)); A.a -= iA * vcross(rA, Pv);
    B.c = vadd(B.c, vmul(mB, Pv)); B.a += iB * vcross(rB, Pv);
    put_pos(t.a, A); put_pos(t.b, B);
    return separation;
  }
  // ---- contacts whose body A is static (walls, boxes): the A side of every
  // solver update is multiplied by invMass = invI = 0, and in the position
  // solver rB == 0 (the manifold point is the circle centre).  Dropping those
  // exact no-ops lets the agent's state stay in registers across iterations;
  // the arithmetic that remains is bit-identical to the generic routines.
  DEV void warm_start_static(f2 normal, f2 rB, float ni_, float ti_, f2& vB, float& wB) {
    f2 tangent = cross_vs(normal, 1.0f);
    f2 Pv = vadd(vmul(ni_, normal), vmul(ti_, tangent));
    wB += C.inv_I * vcross(rB, Pv);
    vB = vadd(vB, vmul(C.inv_mass, Pv));
  }
  DEV void solve_velocity_static(f2 normal, f2 rB, float normalMass, float tangentMass, float& ni_, float& ti_, f2& vB, float& wB) {
    const f2 tangent = cross_vs(normal, 1.0f);
    {
      f2 dv = vadd(vB, cross_sv(wB, rB));
      float vt = vdot(dv, tangent) - 0.0f;
      float lambda = tangentMass * (-vt);
      float maxFriction = C.friction * ni_;
      float newImpulse = fclamp_(ti_ + lambda, -maxFriction, maxFriction);
      lambda = newImpulse - ti_; ti_ = newImpulse;
      f2 Pv = vmul(lambda, tangent);
      vB = vadd(vB, vmul(C.inv_mass, Pv)); wB += C.inv_I * vcross(rB, Pv);
    }
    {
      f2 dv = vadd(vB, cross_sv(wB, rB));
      float vn = vdot(dv, normal);
      float lambda = -normalMass * (vn - 0.0f);
      float newImpulse = fmax_(ni_ + lambda, 0.0f);
      lambda = newImpulse - ni_; ni_ = newImpulse;
      f2 Pv = vmul(lambda, normal);
      vB = vadd(vB, vmul(C.inv_mass, Pv)); wB += C.inv_I * vcross(rB, Pv);
    }
  }
  // init_velocity for a static body A and agent B at cB: world normal, plane
  // point, rB and the effective masses (mA = iA = 0 terms are exact zeros)
  DEV void init_velocity_static(int sid, f2 localNormal, f2 localPoint, f2 cB, f2& normal, f2& planePoint, f2& rB,
                                float& normalMass, float& tangentMass) {
    SBox bx = static_box(sid);
    normal = qmul(bx.qs, bx.qc, localNormal);
    planePoint = sb_mul(bx, localPoint);
    f2 pA = vadd(cB, vmul(B2_POLY_RADIUS - vdot(vsub(cB, planePoint), normal), normal));
    f2 pB = vsub(cB, vmul(C.agent_r, normal));
    f2 point = vmul(0.5f, vadd(pA, pB));
    rB = vsub(point, cB);
    float rnB = vcross(rB, normal);
    float kNormal = C.inv_mass + C.inv_I * rnB * rnB;
    normalMass = kNormal > 0.0f ? 1.0f / kNormal : 0.0f;
    f2 tangent = cross_vs(normal, 1.0f);
    float rtB = vcross(rB, tangent);
    float kTangent = C.inv_mass + C.inv_I * rtB * rtB;
    tangentMass = kTangent > 0.0f ? 1.0f / kTangent : 0.0f;
  }
  // world normal and plane point of a static face contact (constant while solving)
  DEV void static_plane(const TCon& t, f2& normal, f2& planePoint) {
    SBox bx = static_box(t.sid);
    normal = qmul(bx.qs, bx.qc, t.m.localNormal);
    planePoint = sb_mul(bx, t.m.localPoint);
  }
  DEV float solve_position_static(f2 normal, f2 planePoint, f2& cB, bool toi) {
    float separation = vdot(vsub(cB, planePoint), normal) - B2_POLY_RADIUS - C.agent_r;
    float Cc = fclamp_((toi ? B2_TOI_BAUMGARTE : B2_BAUMGARTE) * (separation + B2_LINEAR_SLOP), -B2_MAX_LIN_CORR, 0.0f);
    float K = C.inv_mass;                       // mA + mB + iA*rnA^2 + iB*rnB^2 with mA = iA = 0, rnB = 0
    float impulse = K > 0.0f ? -Cc / K : 0.0f;
    f2 Pv = vmul(impulse, normal);
    cB = vadd(cB, vmul(C.inv_mass, Pv));        // aB += iB * cross(0, P) == aB
    return separation;
  }

  DEV void integrate_position(int i, float h) {  // b2Island::Solve "Integrate positions"
    f2 v = mk2(AG(F_VX, i), AG(F_VY, i)); float w = AG(F_W, i);
    f2 translation = vmul(h, v);
    if (vdot(translation, translation) > B2_MAX_TRANSLATION * B2_MAX_TRANSLATION) {
      float ratio = B2_MAX_TRANSLATION / vlen(translation);
      v = vmul(ratio, v);
    }
    float rotation = h * w;
    if (rotation * rotation > B2_MAX_ROTATION * B2_MAX_ROTATION) {
      float ratio = B2_MAX_ROTATION / fabsf(rotation);
      w *= ratio;
    }
    AG(F_CX, i) += h * v.x; AG(F_CY, i) += h * v.y; AG(F_A, i) += h * w;
    AG(F_VX, i) = v.x; AG(F_VY, i) = v.y; AG(F_W, i) = w;
  }

  // b2Body::SynchronizeFixtures + b2DynamicTree::MoveProxy for agent i
  DEV void synchronize_fixtures(int i) {
    float r = C.agent_r;
    float c0x = AG(F_C0X, i), c0y = AG(F_C0Y, i), cx = AG(F_CX, i), cy = AG(F_CY, i);
    float a1[4] = {c0x - r, c0y - r, c0x + r, c0y + r};
    float a2[4] = {cx - r, cy - r, cx + r, cy + r};
    float ab[4] = {fmin_(a1[0], a2[0]), fmin_(a1[1], a2[1]), fmax_(a1[2], a2[2]), fmax_(a1[3], a2[3])};
    float f0 = AG(F_FAT0, i), f1 = AG(F_FAT1, i), f2_ = AG(F_FAT2, i), f3 = AG(F_FAT3, i);
    if (f0 <= ab[0] && f1 <= ab[1] && ab[2] <= f2_ && ab[3] <= f3) return;
    float n0 = ab[0] - B2_AABB_EXT, n1 = ab[1] - B2_AABB_EXT, n2 = ab[2] + B2_AABB_EXT, n3 = ab[3] + B2_AABB_EXT;
    float dx = B2_AABB_MULT * (cx - c0x), dy = B2_AABB_MULT * (cy - c0y);
    if (dx < 0.0f) n0 += dx; else n2 += dx;
    if (dy < 0.0f) n1 += dy; else n3 += dy;
    AG(F_FAT0, i) = n0; AG(F_FAT1, i) = n1; AG(F_FAT2, i) = n2; AG(F_FAT3, i) = n3;
    AGF(i) |= FL_MOVED;
  }

  // b2Island::Solve for the island of ONE awake agent whose touching contacts
  // are all against static bodies (the usual case).  `ord` lists the contacts
  // (shared-list slots, 5 bits each) in island order = newest first.  With
  // NRr <= NR the contact constants and impulses stay in registers.
  template <int NRr>
  DEV void island_single(int i, int cnt, unsigned long long ord, float h, float dtRatio) {
    f2 cB = apos(i);
    AG(F_C0X, i) = cB.x; AG(F_C0Y, i) = cB.y; AG(F_A0, i) = AG(F_A, i);
    f2 vB = mk2(C.damp * AG(F_VX, i), C.damp * AG(F_VY, i)); float wB = AG(F_W, i) * C.damp;  // v *= 1/(1+h*damping)
    f2 nrm[NRr], pp[NRr];
    bool ok = true;
    if (cnt > 0) {
      f2 rB[NRr]; float nm[NRr], tm[NRr], ni_[NRr], ti_[NRr]; int pr[NRr];
#pragma unroll (NRr <= NR ? NRr : 1)
      for (int k = 0; k < NRr; ++k) {
        if (k < cnt) {
          int s = (int)((ord >> (5 * k)) & 31ull);
          int a_, sid, b_; meta_unpack(KI(K_META, s), pr[k], a_, sid, b_);
          ni_[k] = dtRatio * KF(K_NI, s); ti_[k] = dtRatio * KF(K_TI, s);
          init_velocity_static(sid, mk2(KF(K_LNX, s), KF(K_LNY, s)), mk2(KF(K_LPX, s), KF(K_LPY, s)), cB,
                               nrm[k], pp[k], rB[k], nm[k], tm[k]);
        }
      }
#pragma unroll (NRr <= NR ? NRr : 1)
      for (int k = 0; k < NRr; ++k) if (k < cnt) warm_start_static(nrm[k], rB[k], ni_[k], ti_[k], vB, wB);
      // A sweep is a pure function of (velocity, accumulated impulses): after one that changed none of those bits
      // every further sweep is a no-op, so the loop stops there (the usual case after 1-4 sweeps) -- FIXPOINT_EXIT
      for (int it = 0; it < 10; ++it) {
        const f2 v_in = vB; const float w_in = wB; bool changed = false;
#pragma unroll (NRr <= NR ? NRr : 1)
        for (int k = 0; k < NRr; ++k) if (k < cnt) {
          const float n0 = ni_[k], t0 = ti_[k];
          solve_velocity_static(nrm[k], rB[k], nm[k], tm[k], ni_[k], ti_[k], vB, wB);
          changed |= (__float_as_uint(ni_[k]) != __float_as_uint(n0)) | (__float_as_uint(ti_[k]) != __float_as_uint(t0));
        }
        if (MSV_FIXPOINT && !changed && __float_as_uint(vB.x) == __float_as_uint(v_in.x) && __float_as_uint(vB.y) == __float_as_uint(v_in.y) &&
            __float_as_uint(wB) == __float_as_uint(w_in)) break;
      }
#pragma unroll (NRr <= NR ? NRr : 1)
      for (int k = 0; k < NRr; ++k) if (k < cnt) S.pimp[pr[k] * N + e] = make_float2(ni_[k], ti_[k]);
    }
    AG(F_VX, i) = vB.x; AG(F_VY, i) = vB.y; AG(F_W, i) = wB;
    integrate_position(i, h);
    if (cnt > 0) {
      ok = false;
      cB = apos(i);
      for (int it = 0; it < 10 && !ok; ++it) {
        float minSep = 0.0f;
#pragma unroll (NRr <= NR ? NRr : 1)
        for (int k = 0; k < NRr; ++k) if (k < cnt) minSep = fmin_(minSep, solve_position_static(nrm[k], pp[k], cB, false));
        ok = minSep >= -3.0f * B2_LINEAR_SLOP;
      }
      AG(F_CX, i) = cB.x; AG(F_CY, i) = cB.y;
    }
    {
      const float linTol = B2_LIN_SLEEP_TOL * B2_LIN_SLEEP_TOL, angTol = B2_ANG_SLEEP_TOL * B2_ANG_SLEEP_TOL;
      float w = AG(F_W, i); f2 v = mk2(AG(F_VX, i), AG(F_VY, i));
      float st;
      if (w * w > angTol || vdot(v, v) > linTol) st = 0.0f; else st = AG(F_SLEEP, i) + h;
      AG(F_SLEEP, i) = st;
      if (ok && st >= B2_TIME_TO_SLEEP) sleep_body(i);
    }
    synchronize_fixtures(i);
  }
  // [lane] island of agent i when no agent touches another agent
  DEV void solve_single(int i, float h, float dtRatio) {
    int f = AGF(i);
    if (!(f & FL_ALIVE) || !(f & FL_AWAKE)) return;
    AGF(i) = f | FL_ISLAND;
    // the agent's contact edges, newest (largest creation sequence) first
    unsigned long long ord = 0ull; int cnt = 0; unsigned taken = 0;
    for (;;) {
      int best = -1, bestSeq = -1;
      for (int k = 0; k < ntc; ++k) {
        if ((taken >> k) & 1u) continue;
        int p, a_, sid, b_; meta_unpack(KI(K_META, k), p, a_, sid, b_);
        if (b_ != i || a_ >= 0) continue;
        if (!bit(en, p) || !bit(tc, p)) continue;
        int sq = KI(K_SEQ, k);
        if (sq > bestSeq) { bestSeq = sq; best = k; }
      }
      if (best < 0) break;
      taken |= 1u << best;
      ord |= (unsigned long long)best << (5 * cnt); cnt++;
    }
    SUB_BEGIN();
    if (cnt <= NR) island_single<NR>(i, cnt, ord, h, dtRatio);
    else island_single<BC + 4>(i, cnt, ord, h, dtRatio);
    SUBMAX(cnt <= NR ? 6 : 7, cnt);
  }

  // b2World::Solve for ONE island that contains agent-agent contacts, executed by the lane of the
  // island's seed (the highest-index awake agent of the component: Box2D seeds in body-list order,
  // newest body first): DFS over touching contacts, contact edges newest first, then
  // b2Island::Solve.  Everything lives in the environment's shared-memory column -- body state in
  // the agent fields, solver constants and impulses in the island's own contact-list entries
  // (KS_*) -- so several islands of one environment are solved concurrently by different lanes and
  // nothing goes through local memory.  Contacts against static bodies use the routines that drop
  // the exact no-ops of a massless body A (same arithmetic as the two-body form).
  struct Ord { unsigned long long lo, hi; };   // island contact order: list slots, 5 bits each
  DEV static int ord_get(const Ord& o, int k) { return k < 12 ? (int)((o.lo >> (5 * k)) & 31ull) : (int)((o.hi >> (5 * (k - 12))) & 31ull); }
  DEV static void ord_put(Ord& o, int k, int v) { if (k < 12) o.lo |= (unsigned long long)v << (5 * k); else o.hi |= (unsigned long long)v << (5 * (k - 12)); }
  // b2Island::Solve (after the damping) for an island of exactly TWO agents X < Y with at most NP
  // contacts -- their agent-agent contact plus a few against static bodies -- with the bodies and the
  // contact constants in registers (statically indexed, loops unrolled).  Same arithmetic, same order
  // of operations as the general shared-memory loops of solve_island() below.
  static constexpr int NP = 3;
  DEV void island_pair(unsigned inisl, int nc, const Ord& ord, float h, float dtRatio) {
    const int X = __ffs((int)inisl) - 1, Y = 31 - __clz((int)inisl);
    f2 cX = apos(X), cY = apos(Y);
    f2 vX = mk2(AG(F_VX, X), AG(F_VY, X)), vY = mk2(AG(F_VX, Y), AG(F_VY, Y));
    float wX = AG(F_W, X), wY = AG(F_W, Y), aX = AG(F_A, X), aY = AG(F_A, Y);
    const float mI = C.inv_mass, iI = C.inv_I;
    int ty[NP], pr[NP];                          // 0: X-Y contact, 1: static body vs X, 2: static body vs Y
    f2 nrm[NP], px[NP], rB[NP]; float nm[NP], tm[NP], ni_[NP], ti_[NP];
#pragma unroll
    for (int k = 0; k < NP; ++k) {
      ty[k] = 0; pr[k] = 0; nrm[k] = mk2(0.f, 0.f); px[k] = nrm[k]; rB[k] = nrm[k]; nm[k] = tm[k] = ni_[k] = ti_[k] = 0.0f;
      if (k >= nc) continue;
      const int s = ord_get(ord, k);
      int a_, sid, b_; meta_unpack(KI(K_META, s), pr[k], a_, sid, b_);
      ni_[k] = dtRatio * KF(K_NI, s); ti_[k] = dtRatio * KF(K_TI, s);
      if (a_ >= 0) {   // two dynamic circles (b2WorldManifold::Initialize, e_circles); body A = X, body B = Y
        ty[k] = 0;
        f2 normal = mk2(1.0f, 0.0f);
        if (vlen2(vsub(cX, cY)) > B2_EPS * B2_EPS) { normal = vsub(cY, cX); vnormalize(normal); }
        const f2 pA = vadd(cX, vmul(C.agent_r, normal)), pB = vsub(cY, vmul(C.agent_r, normal));
        const f2 point = vmul(0.5f, vadd(pA, pB));
        px[k] = vsub(point, cX); rB[k] = vsub(point, cY);                  // px := rA
        const float rnA = vcross(px[k], normal), rnB = vcross(rB[k], normal);
        const float kNormal = mI + mI + iI * rnA * rnA + iI * rnB * rnB;
        nm[k] = kNormal > 0.0f ? 1.0f / kNormal : 0.0f;
        const f2 tangent = cross_vs(normal, 1.0f);
        const float rtA = vcross(px[k], tangent), rtB = vcross(rB[k], tangent);
        const float kTangent = mI + mI + iI * rtA * rtA + iI * rtB * rtB;
        tm[k] = kTangent > 0.0f ? 1.0f / kTangent : 0.0f;
        nrm[k] = normal;
      } else {
        ty[k] = b_ == X ? 1 : 2;
        init_velocity_static(sid, mk2(KF(K_LNX, s), KF(K_LNY, s)), mk2(KF(K_LPX, s), KF(K_LPY, s)), b_ == X ? cX : cY,
                             nrm[k], px[k], rB[k], nm[k], tm[k]);           // px := plane point
      }
    }
    for (int it = -1; it < 10; ++it) {           // warm start, then 10 velocity iterations, contacts in island order
      const f2 vX_in = vX, vY_in = vY; const float wX_in = wX, wY_in = wY; bool changed = false;   // FIXPOINT_EXIT (see island_single)
#pragma unroll
      for (int k = 0; k < NP; ++k) {
        if (k >= nc) continue;
        const float n0_ = ni_[k], t0_ = ti_[k];
        if (ty[k] != 0) {
          f2 vB = ty[k] == 1 ? vX : vY; float wB = ty[k] == 1 ? wX : wY;
          if (it < 0) warm_start_static(nrm[k], rB[k], ni_[k], ti_[k], vB, wB);
          else solve_velocity_static(nrm[k], rB[k], nm[k], tm[k], ni_[k], ti_[k], vB, wB);
          if (ty[k] == 1) { vX = vB; wX = wB; } else { vY = vB; wY = wB; }
        } else {
          const f2 normal = nrm[k], rA = px[k], rB_ = rB[k], tangent = cross_vs(normal, 1.0f);
          if (it < 0) {   // b2ContactSolver::WarmStart
            const f2 Pv = vadd(vmul(ni_[k], normal), vmul(ti_[k], tangent));
            wX -= iI * vcross(rA, Pv); vX = vsub(vX, vmul(mI, Pv));
            wY += iI * vcross(rB_, Pv); vY = vadd(vY, vmul(mI, Pv));
          } else {        // b2ContactSolver::SolveVelocityConstraints: friction, then the normal constraint
            {
              const f2 dv = vsub(vsub(vadd(vY, cross_sv(wY, rB_)), vX), cross_sv(wX, rA));
              const float vt = vdot(dv, tangent) - 0.0f;
              float lambda = tm[k] * (-vt);
              const float maxFriction = C.friction * ni_[k];
              const float newImpulse = fclamp_(ti_[k] + lambda, -maxFriction, maxFriction);
              lambda = newImpulse - ti_[k]; ti_[k] = newImpulse;
              const f2 Pv = vmul(lambda, tangent);
              vX = vsub(vX, vmul(mI, Pv)); wX -= iI * vcross(rA, Pv);
              vY = vadd(vY, vmul(mI, Pv)); wY += iI * vcross(rB_, Pv);
            }
            {
              const f2 dv = vsub(vsub(vadd(vY, cross_sv(wY, rB_)), vX), cross_sv(wX, rA));
              const float vn = vdot(dv, normal);
              float lambda = -nm[k] * (vn - 0.0f);
              const float newImpulse = fmax_(ni_[k] + lambda, 0.0f);
              lambda = newImpulse - ni_[k]; ni_[k] = newImpulse;
              const f2 Pv = vmul(lambda, normal);
              vX = vsub(vX, vmul(mI, Pv)); wX -= iI * vcross(rA, Pv);
              vY = vadd(vY, vmul(mI, Pv)); wY += iI * vcross(rB_, Pv);
            }
          }
        }
        changed |= (__float_as_uint(ni_[k]) != __float_as_uint(n0_)) | (__float_as_uint(ti_[k]) != __float_as_uint(t0_));
      }
      if (MSV_FIXPOINT && it >= 0 && !changed &&
          __float_as_uint(vX.x) == __float_as_uint(vX_in.x) && __float_as_uint(vX.y) == __float_as_uint(vX_in.y) && __float_as_uint(wX) == __float_as_uint(wX_in) &&
          __float_as_uint(vY.x) == __float_as_uint(vY_in.x) && __float_as_uint(vY.y) == __float_as_uint(vY_in.y) && __float_as_uint(wY) == __float_as_uint(wY_in)) break;
    }
#pragma unroll
    for (int k = 0; k < NP; ++k) if (k < nc) S.pimp[pr[k] * N + e] = make_float2(ni_[k], ti_[k]);   // b2ContactSolver::StoreImpulses
    AG(F_VX, X) = vX.x; AG(F_VY, X) = vX.y; AG(F_W, X) = wX; AG(F_VX, Y) = vY.x; AG(F_VY, Y) = vY.y; AG(F_W, Y) = wY;
    integrate_position(X, h); integrate_position(Y, h);
    cX = apos(X); cY = apos(Y); aX = AG(F_A, X); aY = AG(F_A, Y);
    bool ok = false;
    for (int it = 0; it < 10 && !ok; ++it) {     // b2ContactSolver::SolvePositionConstraints
      float minSep = 0.0f;
#pragma unroll
      for (int k = 0; k < NP; ++k) {
        if (k >= nc) continue;
        float separation;
        if (ty[k] == 1) separation = solve_position_static(nrm[k], px[k], cX, false);
        else if (ty[k] == 2) separation = solve_position_static(nrm[k], px[k], cY, false);
        else {         // circles: the manifold point is the midpoint, normal along the centres
          f2 normal = vsub(cY, cX); vnormalize(normal);
          const f2 point = vmul(0.5f, vadd(cX, cY));
          separation = vdot(vsub(cY, cX), normal) - C.agent_r - C.agent_r;
          const f2 rA = vsub(point, cX), rB_ = vsub(point, cY);
          const float Cc = fclamp_(B2_BAUMGARTE * (separation + B2_LINEAR_SLOP), -B2_MAX_LIN_CORR, 0.0f);
          const float rnA = vcross(rA, normal), rnB = vcross(rB_, normal);
          const float K = mI + mI + iI * rnA * rnA + iI * rnB * rnB;
          const float impulse = K > 0.0f ? -Cc / K : 0.0f;
          const f2 Pv = vmul(impulse, normal);
          cX = vsub(cX, vmul(mI, Pv)); aX -= iI * vcross(rA, Pv);
          cY = vadd(cY, vmul(mI, Pv)); aY += iI * vcross(rB_, Pv);
        }
        minSep = fmin_(minSep, separation);
      }
      ok = minSep >= -3.0f * B2_LINEAR_SLOP;
    }
    AG(F_CX, X) = cX.x; AG(F_CY, X) = cX.y; AG(F_A, X) = aX; AG(F_CX, Y) = cY.x; AG(F_CY, Y) = cY.y; AG(F_A, Y) = aY;
    {
      const float linTol = B2_LIN_SLEEP_TOL * B2_LIN_SLEEP_TOL, angTol = B2_ANG_SLEEP_TOL * B2_ANG_SLEEP_TOL;
      bool can_sleep = ok;                       // minSleepTime >= timeToSleep && positionSolved
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const int i = q == 0 ? X : Y;
        float w = AG(F_W, i); f2 v = mk2(AG(F_VX, i), AG(F_VY, i));
        float st;
        if (w * w > angTol || vdot(v, v) > linTol) st = 0.0f; else st = AG(F_SLEEP, i) + h;
        AG(F_SLEEP, i) = st;
        if (!(st >= B2_TIME_TO_SLEEP)) can_sleep = false;
      }
      if (can_sleep) { sleep_body(X); sleep_body(Y); }
    }
    synchronize_fixtures(X); synchronize_fixtures(Y);
  }
  COLD0 void solve_island(int seed, float h, float dtRatio) {
    SUB_BEGIN();
    Ord ord; ord.lo = 0ull; ord.hi = 0ull;
    int nc = 0; unsigned taken = 0, inisl = 1u << seed;
    {
      unsigned stack = (unsigned)seed; int sc = 1;    // agent indices, 4 bits each
      AGF(seed) |= FL_ISLAND;
      while (sc > 0) {
        --sc;
        const int bI = (int)((stack >> (4 * sc)) & 15u);
        wake(bI);
        for (;;) {  // contact edges of bI, newest (largest seq) first
          int best = -1, bestSeq = -1, bestMeta = 0;
          for (int k = 0; k < ntc; ++k) {
            if ((taken >> k) & 1u) continue;
            const int meta = KI(K_META, k);
            int p, a_, sid, b_; meta_unpack(meta, p, a_, sid, b_);
            if (a_ != bI && b_ != bI) continue;
            if (!bit(en, p) || !bit(tc, p)) continue;
            const int sq = KI(K_SEQ, k);
            if (sq > bestSeq) { bestSeq = sq; best = k; bestMeta = meta; }
          }
          if (best < 0) break;
          taken |= 1u << best;
          ord_put(ord, nc, best); nc++;
          int p, a_, sid, b_; meta_unpack(bestMeta, p, a_, sid, b_);
          if (a_ >= 0) {
            const int other = a_ == bI ? b_ : a_;
            if (!(AGF(other) & FL_ISLAND)) {
              stack = (stack & ~(15u << (4 * sc))) | ((unsigned)other << (4 * sc)); sc++;
              AGF(other) |= FL_ISLAND; inisl |= 1u << other;
            }
          }
        }
      }
    }
    // ---- b2Island::Solve
    for (int i = 0; i < C.A; ++i) {
      if (!((inisl >> i) & 1u)) continue;
      AG(F_C0X, i) = AG(F_CX, i); AG(F_C0Y, i) = AG(F_CY, i); AG(F_A0, i) = AG(F_A, i);
      AG(F_VX, i) = C.damp * AG(F_VX, i); AG(F_VY, i) = C.damp * AG(F_VY, i);  // v *= 1/(1+h*damping)
      AG(F_W, i) *= C.damp;
    }
    SUB(8);
    if (__popc(inisl) == 2 && nc <= NP) { island_pair(inisl, nc, ord, h, dtRatio); SUB(9); return; }   // two agents, <= NP contacts (the usual case)
    SUBCNT(14, 1); SUBCNT(15, nc);
    // b2ContactSolver::InitializeVelocityConstraints (+ the warm-start scaling of b2ContactSolver's constructor)
    for (int k = 0; k < nc; ++k) {
      const int s = ord_get(ord, k);
      int p, a_, sid, b_; meta_unpack(KI(K_META, s), p, a_, sid, b_);
      const f2 ln = mk2(KF(K_LNX, s), KF(K_LNY, s)), lp = mk2(KF(K_LPX, s), KF(K_LPY, s));
      KF(K_NI, s) = dtRatio * KF(K_NI, s); KF(K_TI, s) = dtRatio * KF(K_TI, s);
      f2 normal, px, rB; float nm, tm;
      if (a_ >= 0) {   // two dynamic circles (b2WorldManifold::Initialize, e_circles)
        const f2 cA = apos(a_), cB = apos(b_);
        normal = mk2(1.0f, 0.0f);
        if (vlen2(vsub(cA, cB)) > B2_EPS * B2_EPS) { normal = vsub(cB, cA); vnormalize(normal); }
        const f2 pA = vadd(cA, vmul(C.agent_r, normal)), pB = vsub(cB, vmul(C.agent_r, normal));
        const f2 point = vmul(0.5f, vadd(pA, pB));
        px = vsub(point, cA); rB = vsub(point, cB);                      // px := rA
        const float rnA = vcross(px, normal), rnB = vcross(rB, normal);
        const float kNormal = C.inv_mass + C.inv_mass + C.inv_I * rnA * rnA + C.inv_I * rnB * rnB;
        nm = kNormal > 0.0f ? 1.0f / kNormal : 0.0f;
        const f2 tangent = cross_vs(normal, 1.0f);
        const float rtA = vcross(px, tangent), rtB = vcross(rB, tangent);
        const float kTangent = C.inv_mass + C.inv_mass + C.inv_I * rtA * rtA + C.inv_I * rtB * rtB;
        tm = kTangent > 0.0f ? 1.0f / kTangent : 0.0f;
      } else {
        init_velocity_static(sid, ln, lp, apos(b_), normal, px, rB, nm, tm);   // px := plane point
      }
      KF(KS_NX, s) = normal.x; KF(KS_NY, s) = normal.y; KF(KS_PX, s) = px.x; KF(KS_PY, s) = px.y;
      KF(KS_RBX, s) = rB.x; KF(KS_RBY, s) = rB.y; KF(K_NM, s) = nm; KF(K_TM, s) = tm;
    }
    SUB(10);
    // warm start, then 10 velocity iterations, contacts in island order.  The bodies' velocities (then positions)
    // live in REGISTERS -- one record per agent slot, picked with statically unrolled selects -- because the
    // Gauss-Seidel sweep is one long dependent chain through them: a shared-memory store/load round trip per
    // contact and iteration is what made a 4-agent pile-up cost ~100k cycles.  The per-contact constants, which
    // are off that chain, stay in shared memory.
    f2 bv[AC]; float bw[AC];
#pragma unroll
    for (int q = 0; q < AC; ++q) { bv[q] = mk2(AG(F_VX, q), AG(F_VY, q)); bw[q] = AG(F_W, q); }
    auto getv = [&](int i, f2& v, float& w) {
      v = bv[0]; w = bw[0];
#pragma unroll
      for (int q = 1; q < AC; ++q) if (i == q) { v = bv[q]; w = bw[q]; }
    };
    auto setv = [&](int i, f2 v, float w) {
#pragma unroll
      for (int q = 0; q < AC; ++q) if (i == q) { bv[q] = v; bw[q] = w; }
    };
    for (int it = -1; it < 10; ++it) {
      for (int k = 0; k < nc; ++k) {
        const int s = ord_get(ord, k);
        int p, a_, sid, b_; meta_unpack(KI(K_META, s), p, a_, sid, b_);
        const f2 normal = mk2(KF(KS_NX, s), KF(KS_NY, s)), rB = mk2(KF(KS_RBX, s), KF(KS_RBY, s));
        const float nm_ = KF(K_NM, s), tm_ = KF(K_TM, s);
        float ni_ = KF(K_NI, s), ti_ = KF(K_TI, s);
        f2 vB; float wB; getv(b_, vB, wB);
        if (a_ < 0) {
          if (it < 0) warm_start_static(normal, rB, ni_, ti_, vB, wB);
          else solve_velocity_static(normal, rB, nm_, tm_, ni_, ti_, vB, wB);
        } else {
          const f2 rA = mk2(KF(KS_PX, s), KF(KS_PY, s)), tangent = cross_vs(normal, 1.0f);
          f2 vA; float wA; getv(a_, vA, wA);
          const float mA = C.inv_mass, iA = C.inv_I, mB = C.inv_mass, iB = C.inv_I;
          if (it < 0) {   // b2ContactSolver::WarmStart
            const f2 Pv = vadd(vmul(ni_, normal), vmul(ti_, tangent));
            wA -= iA * vcross(rA, Pv); vA = vsub(vA, vmul(mA, Pv));
            wB += iB * vcross(rB, Pv); vB = vadd(vB, vmul(mB, Pv));
          } else {        // b2ContactSolver::SolveVelocityConstraints: friction, then the normal constraint
            {
              const f2 dv = vsub(vsub(vadd(vB, cross_sv(wB, rB)), vA), cross_sv(wA, rA));
              const float vt = vdot(dv, tangent) - 0.0f;
              float lambda = tm_ * (-vt);
              const float maxFriction = C.friction * ni_;
              const float newImpulse = fclamp_(ti_ + lambda, -maxFriction, maxFriction);
              lambda = newImpulse - ti_; ti_ = newImpulse;
              const f2 Pv = vmul(lambda, tangent);
              vA = vsub(vA, vmul(mA, Pv)); wA -= iA * vcross(rA, Pv);
              vB = vadd(vB, vmul(mB, Pv)); wB += iB * vcross(rB, Pv);
            }
            {
              const f2 dv = vsub(vsub(vadd(vB, cross_sv(wB, rB)), vA), cross_sv(wA, rA));
              const float vn = vdot(dv, normal);
              float lambda = -nm_ * (vn - 0.0f);
              const float newImpulse = fmax_(ni_ + lambda, 0.0f);
              lambda = newImpulse - ni_; ni_ = newImpulse;
              const f2 Pv = vmul(lambda, normal);
              vA = vsub(vA, vmul(mA, Pv)); wA -= iA * vcross(rA, Pv);
              vB = vadd(vB, vmul(mB, Pv)); wB += iB * vcross(rB, Pv);
            }
          }
          setv(a_, vA, wA);
        }
        setv(b_, vB, wB);
        KF(K_NI, s) = ni_; KF(K_TI, s) = ti_;
      }
    }
#pragma unroll
    for (int q = 0; q < AC; ++q) if ((inisl >> q) & 1u) { AG(F_VX, q) = bv[q].x; AG(F_VY, q) = bv[q].y; AG(F_W, q) = bw[q]; }
    for (int k = 0; k < nc; ++k) {   // b2ContactSolver::StoreImpulses
      const int s = ord_get(ord, k);
      S.pimp[(KI(K_META, s) & 255) * N + e] = make_float2(KF(K_NI, s), KF(K_TI, s));
    }
    SUB(11);
    for (int i = 0; i < C.A; ++i) if ((inisl >> i) & 1u) integrate_position(i, h);
    // positions: the same register scheme (bv := centre, bw := angle)
#pragma unroll
    for (int q = 0; q < AC; ++q) { bv[q] = mk2(AG(F_CX, q), AG(F_CY, q)); bw[q] = AG(F_A, q); }
    bool ok = false;
    for (int it = 0; it < 10 && !ok; ++it) {   // b2ContactSolver::SolvePositionConstraints
      float minSep = 0.0f;
      for (int k = 0; k < nc; ++k) {
        const int s = ord_get(ord, k);
        int p, a_, sid, b_; meta_unpack(KI(K_META, s), p, a_, sid, b_);
        f2 cB; float aB; getv(b_, cB, aB);
        float separation;
        if (a_ < 0) {
          separation = solve_position_static(mk2(KF(KS_NX, s), KF(KS_NY, s)), mk2(KF(KS_PX, s), KF(KS_PY, s)), cB, false);
        } else {       // circles: the manifold point is the midpoint, normal along the centres
          f2 cA; float aA; getv(a_, cA, aA);
          const float mA = C.inv_mass, iA = C.inv_I, mB = C.inv_mass, iB = C.inv_I;
          f2 normal = vsub(cB, cA); vnormalize(normal);
          const f2 point = vmul(0.5f, vadd(cA, cB));
          separation = vdot(vsub(cB, cA), normal) - C.agent_r - C.agent_r;
          const f2 rA = vsub(point, cA), rB = vsub(point, cB);
          const float Cc = fclamp_(B2_BAUMGARTE * (separation + B2_LINEAR_SLOP), -B2_MAX_LIN_CORR, 0.0f);
          const float rnA = vcross(rA, normal), rnB = vcross(rB, normal);
          const float K = mA + mB + iA * rnA * rnA + iB * rnB * rnB;
          const float impulse = K > 0.0f ? -Cc / K : 0.0f;
          const f2 Pv = vmul(impulse, normal);
          cA = vsub(cA, vmul(mA, Pv)); aA -= iA * vcross(rA, Pv);
          cB = vadd(cB, vmul(mB, Pv)); aB += iB * vcross(rB, Pv);
          setv(a_, cA, aA);
        }
        setv(b_, cB, aB);
        minSep = fmin_(minSep, separation);
      }
      ok = minSep >= -3.0f * B2_LINEAR_SLOP;
    }
#pragma unroll
    for (int q = 0; q < AC; ++q) if ((inisl >> q) & 1u) { AG(F_CX, q) = bv[q].x; AG(F_CY, q) = bv[q].y; AG(F_A, q) = bw[q]; }
    SUB(12);
    {
      const float linTol = B2_LIN_SLEEP_TOL * B2_LIN_SLEEP_TOL, angTol = B2_ANG_SLEEP_TOL * B2_ANG_SLEEP_TOL;
      bool can_sleep = ok;                       // minSleepTime >= timeToSleep && positionSolved
      for (int i = 0; i < C.A; ++i) {
        if (!((inisl >> i) & 1u)) continue;
        float w = AG(F_W, i); f2 v = mk2(AG(F_VX, i), AG(F_VY, i));
        float st;
        if (w * w > angTol || vdot(v, v) > linTol) st = 0.0f; else st = AG(F_SLEEP, i) + h;
        AG(F_SLEEP, i) = st;
        if (!(st >= B2_TIME_TO_SLEEP)) can_sleep = false;
      }
      if (can_sleep)
        for (int i = 0; i < C.A; ++i) if ((inisl >> i) & 1u) sleep_body(i);
    }
    for (int i = 0; i < C.A; ++i)
      if ((inisl >> i) & 1u) synchronize_fixtures(i);
  }

  // b2World::Solve                                                   [all lanes]
  // Agents with a touching, enabled agent-agent contact form islands of several bodies: each such
  // island is solved by the lane of its seed agent (solve_island); every other awake agent is an
  // island of its own, solved by its lane (solve_single).
  __device__ __forceinline__ void solve(float h, float dtRatio) {
    unsigned awk = 0;
    for (int i = g; i < C.A; i += G) { AGF(i) &= ~(FL_ISLAND | FL_MOVED); if ((AGF(i) & (FL_ALIVE | FL_AWAKE)) == (FL_ALIVE | FL_AWAKE)) awk |= 1u << i; }
    unsigned long long aa = tc[0] & en[0]; if (NAA < 64) aa &= (1ull << NAA) - 1ull;   // touching agent-agent pairs
    awk = or32(awk);                           // one consistent snapshot of the awake flags (islands wake bodies)
    gsync();
    for (int i = g; i < C.A; i += G) {
      if (aa == 0ull) { solve_single(i, h, dtRatio); continue; }    // group-uniform: nobody touches another agent
      // connected component of agent i over the touching agent-agent contacts
      unsigned comp = 1u << i;
      for (int it = 0; it < AC; ++it) {
        unsigned grown = comp;
        for (int j = 0; j < C.A; ++j) {
          if (!((comp >> j) & 1u)) continue;
          for (int a = 0; a < j; ++a) if ((aa >> p_aa(a, j)) & 1ull) grown |= 1u << a;
          for (int b = j + 1; b < C.A; ++b) if ((aa >> p_aa(j, b)) & 1ull) grown |= 1u << b;
        }
        if (grown == comp) break;
        comp = grown;
      }
      if (comp == (1u << i)) { solve_single(i, h, dtRatio); continue; }
      const unsigned cand = comp & awk;          // no awake member: the island is not simulated
      if (cand != 0u && (31 - __clz((int)cand)) == i) { RARE_BEGIN(); SUB_BEGIN(); MSV_COLDK(0, solve_island(i, h, dtRatio)); SUBMAX(13, __popc(comp)); RARE_END(0); }
    }
    gsync();
  }
  // b2ContactManager::FindNewContacts after the solve (the kernel puts a phase barrier in between)
  __device__ __forceinline__ void solve_find_new() {
    unsigned mv = 0;
    for (int i = g; i < C.A; i += G) if (AGF(i) & FL_MOVED) mv = 1u;
    if (or32(mv)) find_new_contacts(true);
  }

  // b2Body::Advance for agent i
  DEV void advance(int i, float alpha) {
    float a0 = AG(F_ALPHA0, i);
    float beta = (alpha - a0) / (1.0f - a0);
    AG(F_C0X, i) += beta * (AG(F_CX, i) - AG(F_C0X, i));
    AG(F_C0Y, i) += beta * (AG(F_CY, i) - AG(F_C0Y, i));
    AG(F_A0, i) += beta * (AG(F_A, i) - AG(F_A0, i));
    AG(F_ALPHA0, i) = alpha;
    AG(F_CX, i) = AG(F_C0X, i); AG(F_CY, i) = AG(F_C0Y, i); AG(F_A, i) = AG(F_A0, i);
  }

  // [leader] one TOI event of b2World::SolveTOI on contact minP at minAlpha.
  // Returns bit 0: the contact was touching at the TOI (the sub-step ran);
  // bit 1: the event left everything exactly as the previous one on minP did.
  // The mini island (the TOI contact, then the agent's other touching contacts against static
  // bodies, newest first) keeps its solver constants in the dead touching-contact list (KS_* words of
  // slots 0..TOI_ISL-1; the list is rebuilt by the next Collide), the state snapshot of the previous
  // event in slots 8.., so nothing of the event goes through local memory.
  static constexpr int SNAPW = F_COUNT + 6 * PW + 1;
  static constexpr int TOI_ISL = 8;
  static_assert(SNAPW <= K_COUNT * (MAXC - TOI_ISL), "snapshot does not fit the scratch slots");
  DEV unsigned& SNAP(int q) { CHK((unsigned)q < (unsigned)SNAPW); return reinterpret_cast<unsigned*>(msv_sm)[sb + (W_TC + (q / (MAXC - TOI_ISL)) * MAXC + TOI_ISL + q % (MAXC - TOI_ISL))]; }
  COLD1 int toi_event(int minP, float minAlpha, float dt, int prevP) {
    SUB_BEGIN();
    int a, sid, b; decode(minP, a, sid, b);
    // backup the agent's sweep, advance to the TOI, re-evaluate the contact
    const float bk0 = AG(F_C0X, b), bk1 = AG(F_C0Y, b), bk2 = AG(F_CX, b), bk3 = AG(F_CY, b), bk4 = AG(F_A0, b), bk5 = AG(F_A, b), bk6 = AG(F_ALPHA0, b);
    advance(b, minAlpha);
    int nisl = 0;
    auto isl_add = [&](int sid_, const Manifold& m) {   // world normal and plane point of the face contact (constant while solving)
      SBox bx = static_box(sid_);
      const f2 normal = qmul(bx.qs, bx.qc, m.localNormal), planePoint = sb_mul(bx, m.localPoint);
      KF(KS_NX, nisl) = normal.x; KF(KS_NY, nisl) = normal.y; KF(KS_PX, nisl) = planePoint.x; KF(KS_PY, nisl) = planePoint.y;
      nisl++;
    };
    {
      Manifold m_min; unsigned wk = 0;
      bool touching = contact_update(minP, a, sid, b, false, wk, &m_min);
      wake_all(wk);
      if (!touching) {
        clrb(en, minP);
        AG(F_C0X, b) = bk0; AG(F_C0Y, b) = bk1; AG(F_CX, b) = bk2; AG(F_CY, b) = bk3;
        AG(F_A0, b) = bk4; AG(F_A, b) = bk5; AG(F_ALPHA0, b) = bk6;
        return 0;
      }
      wake(b);
      isl_add(sid, m_min);
    }
    SUB(0);
    {
      // the agent's other existing contacts against static bodies, newest (largest creation sequence) first;
      // the sequence numbers are fetched together (one memory latency), then ranked in registers
      int sq[BC + 4];
#pragma unroll
      for (int k = 0; k < BC + 4; ++k) {
        const int p = k < BC ? p_ab(b, k) : p_aw(b, k - BC);
        sq[k] = ((k < BC && k >= nb) || p == minP || !bit(ex, p)) ? -1 : (int)S.pseq[p * N + e];
      }
      for (;;) {
        int best = -1, bestSeq = -1;
#pragma unroll
        for (int k = 0; k < BC + 4; ++k) if (sq[k] > bestSeq) { bestSeq = sq[k]; best = k; }
        if (best < 0) break;
#pragma unroll
        for (int k = 0; k < BC + 4; ++k) if (k == best) sq[k] = -1;
        if (nisl >= TOI_ISL) { LI(L_OVERFLOW)++; break; }
        const int p2 = best < BC ? p_ab(b, best) : p_aw(b, best - BC);
        Manifold m; unsigned wk2 = 0;
        bool t2 = contact_update(p2, -1, best, b, false, wk2, &m);
        wake_all(wk2);
        if (t2) isl_add(best, m);
      }
    }
    SUB(1);
    const float subdt = (1.0f - minAlpha) * dt;
    // b2Island::SolveTOI -- every contact of the mini island has a static body A
    {
      // A sweep is a pure function of the centre: one that leaves it bitwise unchanged (an agent wedged between
      // opposing faces: the corrections cancel exactly) would repeat verbatim until the iteration limit -> stop there.
      f2 cB = apos(b);
      for (int it = 0; it < 20; ++it) {
        const f2 c_in = cB;
        float minSep = 0.0f;
        for (int k = 0; k < nisl; ++k)
          minSep = fmin_(minSep, solve_position_static(mk2(KF(KS_NX, k), KF(KS_NY, k)), mk2(KF(KS_PX, k), KF(KS_PY, k)), cB, true));
        if (minSep >= -1.5f * B2_LINEAR_SLOP) break;
        if (__float_as_uint(cB.x) == __float_as_uint(c_in.x) && __float_as_uint(cB.y) == __float_as_uint(c_in.y)) break;
      }
      AG(F_CX, b) = cB.x; AG(F_CY, b) = cB.y;
    }
    AG(F_C0X, b) = AG(F_CX, b); AG(F_C0Y, b) = AG(F_CY, b); AG(F_A0, b) = AG(F_A, b);
    SUB(2);
    {
      // b2ContactSolver::InitializeVelocityConstraints at the corrected position (impulses start at zero, no warm start)
      const f2 cB = apos(b);
      for (int k = 0; k < nisl; ++k) {
        const f2 normal = mk2(KF(KS_NX, k), KF(KS_NY, k)), planePoint = mk2(KF(KS_PX, k), KF(KS_PY, k));
        const f2 pA = vadd(cB, vmul(B2_POLY_RADIUS - vdot(vsub(cB, planePoint), normal), normal));
        const f2 pB = vsub(cB, vmul(C.agent_r, normal));
        const f2 point = vmul(0.5f, vadd(pA, pB));
        const f2 rB = vsub(point, cB);
        const float rnB = vcross(rB, normal);
        const float kNormal = C.inv_mass + C.inv_I * rnB * rnB;
        const f2 tangent = cross_vs(normal, 1.0f);
        const float rtB = vcross(rB, tangent);
        const float kTangent = C.inv_mass + C.inv_I * rtB * rtB;
        KF(KS_RBX, k) = rB.x; KF(KS_RBY, k) = rB.y;
        KF(K_NM, k) = kNormal > 0.0f ? 1.0f / kNormal : 0.0f; KF(K_TM, k) = kTangent > 0.0f ? 1.0f / kTangent : 0.0f;
        KF(K_NI, k) = 0.0f; KF(K_TI, k) = 0.0f;
      }
      // Gauss-Seidel sweeps are a pure function of (velocity, accumulated impulses): after a sweep that changed none
      // of those bits every further sweep is a no-op -> stop (the usual case after 1-3 sweeps)
      f2 vB = mk2(AG(F_VX, b), AG(F_VY, b)); float wB = AG(F_W, b);
      for (int it = 0; it < 10; ++it) {
        const f2 v_in = vB; const float w_in = wB; bool changed = false;
        for (int k = 0; k < nisl; ++k) {
          const float ni0 = KF(K_NI, k), ti0 = KF(K_TI, k);
          float ni_ = ni0, ti_ = ti0;
          solve_velocity_static(mk2(KF(KS_NX, k), KF(KS_NY, k)), mk2(KF(KS_RBX, k), KF(KS_RBY, k)), KF(K_NM, k), KF(K_TM, k), ni_, ti_, vB, wB);
          KF(K_NI, k) = ni_; KF(K_TI, k) = ti_;
          changed |= __float_as_uint(ni_) != __float_as_uint(ni0) || __float_as_uint(ti_) != __float_as_uint(ti0);
        }
        if (!changed && __float_as_uint(vB.x) == __float_as_uint(v_in.x) && __float_as_uint(vB.y) == __float_as_uint(v_in.y) &&
            __float_as_uint(wB) == __float_as_uint(w_in)) break;
      }
      AG(F_VX, b) = vB.x; AG(F_VY, b) = vB.y; AG(F_W, b) = wB;
    }
    SUB(3);
    integrate_position(b, subdt);
    AGF(b) &= ~FL_MOVED;
    synchronize_fixtures(b);
    if (AGF(b) & FL_MOVED) find_new_contacts_of(b);
    SUB(4);
    // A TOI event is a pure function of (agent b's sweep/velocity/AABB words, the pair
    // bit-matrices, the contact counter).  If this event left all of them exactly as the
    // previous event on the same contact did, every further event on it would repeat
    // verbatim and only count up to b2_maxSubSteps (a body wedged between two static
    // bodies does this): the caller jumps the contact's toiCount there instead of replaying them.
    bool same = prevP == minP;
    auto snap = [&](int q, unsigned v) { if (SNAP(q) != v) same = false; SNAP(q) = v; };
    for (int f = 0; f < F_COUNT; ++f) snap(f, __float_as_uint(AG(f, b)));
#pragma unroll
    for (int w = 0; w < PW; ++w) {
      snap(F_COUNT + 6 * w + 0, (unsigned)ex[w]); snap(F_COUNT + 6 * w + 1, (unsigned)(ex[w] >> 32));
      snap(F_COUNT + 6 * w + 2, (unsigned)tc[w]); snap(F_COUNT + 6 * w + 3, (unsigned)(tc[w] >> 32));
      snap(F_COUNT + 6 * w + 4, (unsigned)en[w]); snap(F_COUNT + 6 * w + 5, (unsigned)(en[w] >> 32));
    }
    snap(SNAPW - 1, (unsigned)LI(L_CONTACTSEQ));
    SUB(5);
    return 1 | (same ? 2 : 0);
  }

  // b2World::SolveTOI: continuous collision of agents against static boxes
  // and walls (agent-agent pairs are "two non-bullet dynamic bodies": skipped).
  // Every lane evaluates b2TimeOfImpact for the contacts of its own agents;
  // the group picks the minimum; the leader runs the event.
  DEV void solve_toi(float dt) {
    static_assert(SLOTS == 1, "solve_toi: one agent per lane");
    const int i = g;                           // this lane's agent
    if (i < C.A) { AGF(i) &= ~FL_ISLAND; AG(F_ALPHA0, i) = 0.0f; }
    // Per static body k of the lane's agent: the contact's toiCount (4 bits each) and the validity bit of
    // its cached TOI (b2Contact::e_toiFlag / m_toi, the value sits in shared memory); both are only ever
    // needed by the lane that owns the agent.
    unsigned long long evcnt = 0ull; unsigned cvalid = 0u;
    int prevP = -1;                            // leader: contact of the previous event that ran (its state snapshot sits in shared memory)
    // b2TimeOfImpact(static body k, agent j) as SolveTOI evaluates it for a contact without a cached TOI
    auto toi_alpha = [&](int j, int k) {
      const SBox sbx = static_box(k);
      const f2 q0 = mk2(AG(F_C0X, j), AG(F_C0Y, j)), q1 = apos(j);
      float beta = 1.0f;
      const int state = time_of_impact(sbx, q0, q1, C.agent_r, beta);
      const float alpha0 = AG(F_ALPHA0, j);
      return state == TOI_TOUCHING ? fmin_(alpha0 + (1.0f - alpha0) * beta, 1.0f) : 1.0f;
    };
    TOIPROF(long long tp0 = clock64(); long long tp_ev = 0; int tp_it = 0; int tp_ran = 0; int tp_not = 0; int tp_same = 0; int tp_calls = 0;)
    for (int guard = 0; guard < 64; ++guard) {
      TOIPROF(tp_it++;)
      // ---- (1) every lane: the existing, enabled agent-vs-static contacts of its agent that still take part.
      // Cached TOIs enter the minimum directly; the contacts whose TOI must be computed are collected in `need`
      // (bit k = static body k).
      unsigned need = 0u;
      int minP = -1, minSeq = -1; float minAlpha = 1.0f;
      // the world contact list is newest first and the scan keeps the FIRST minimum:
      // on equal alpha the contact with the larger creation sequence wins
      auto consider = [&](int p, float alpha) {
        if (alpha < 1.0f) {
          const int sq = (int)S.pseq[p * N + e];
          if (alpha < minAlpha || (alpha == minAlpha && sq > minSeq)) { minAlpha = alpha; minP = p; minSeq = sq; }
        }
      };
      if (i < C.A && alive(i) && awake(i)) {
#pragma unroll
        for (int w = 0; w < PW; ++w) {
          unsigned long long mbits = ex[w] & en[w] & own[w];
          if (w == 0) mbits &= ~((1ull << NAA) - 1ull);     // pair index >= NAA: against static bodies
          while (mbits) {
            int p = w * 64 + __ffsll((long long)mbits) - 1; mbits &= mbits - 1;
            int a_, k, i_; decode(p, a_, k, i_);
            const int cnt = (int)((evcnt >> (4 * k)) & 15ull);
            if (cnt > C.toi_max_count) continue;       // b2_maxSubSteps (">=" under MSV_B2_SUBSTEPS_GE)
            if ((cvalid >> k) & 1u) { consider(p, TOIA(i, k)); continue; }
            // b2TimeOfImpact can only report e_touching at a time where the true distance
            // between the core shapes is below target + tolerance (0.49625).  The sweep is a
            // straight segment against a static box, so if a lower bound of the segment-box
            // distance (largest per-axis gap in the box frame) clears that with margin, the
            // outcome is alpha = 1 whatever path the root finder takes: skip the call.
            const SBox sbx = static_box(k);
            const f2 l0 = sb_mulT(sbx, mk2(AG(F_C0X, i), AG(F_C0Y, i))), l1 = sb_mulT(sbx, apos(i));
            const float gx = fmax_(fmin_(l0.x, l1.x) - sbx.hx, -sbx.hx - fmax_(l0.x, l1.x));
            const float gy = fmax_(fmin_(l0.y, l1.y) - sbx.hy, -sbx.hy - fmax_(l0.y, l1.y));
            if (fmax_(gx, gy) > (B2_POLY_RADIUS + C.agent_r - 3.0f * B2_LINEAR_SLOP) + 0.25f * B2_LINEAR_SLOP + 0.004f) { TOIA(i, k) = 1.0f; cvalid |= 1u << k; }
            else if (MSV_TOI_COOP) need |= 1u << k;
            else { const float al = toi_alpha(i, k); TOIA(i, k) = al; cvalid |= 1u << k; consider(p, al); }
          }
        }
      }
      // ---- (2) the group computes the missing TOIs together: the calls are dealt out to the lanes in
      // (agent, static body) order, so an agent wedged between several bodies does not serialise them on
      // its own lane while the others idle.  Any lane can evaluate any pair: the inputs sit in shared memory.
      if (MSV_TOI_COOP && __any_sync(gmask, need != 0u)) {          // group-uniform
        unsigned ms[G]; int T = 0;
#pragma unroll
        for (int j = 0; j < G; ++j) { ms[j] = from(need, j); T += __popc(ms[j]); }
        TOIPROF(tp_calls += T;)
        for (int r0 = 0; r0 < T; r0 += G) {
          const int t = r0 + g;
          int fj = -1, fk = 0, base = 0;
#pragma unroll
          for (int j = 0; j < G; ++j) {
            const int c = __popc(ms[j]);
            if (t >= base && t < base + c) { fj = j; fk = (int)__fns(ms[j], 0u, t - base + 1); }
            base += c;
          }
          if (fj >= 0) TOIA(fj, fk) = toi_alpha(fj, fk);
        }
        gsync();
        cvalid |= need;
        while (need) {
          const int k = __ffs((int)need) - 1; need &= need - 1u;
          consider(k < BC ? p_ab(i, k) : p_aw(i, k - BC), TOIA(i, k));
        }
      }
      // ---- (3) minimum over the group
#pragma unroll
      for (int o = 1; o < G; o <<= 1) {        // group minimum (alpha ascending, creation sequence descending)
        float oa = __shfl_xor_sync(gmask, minAlpha, o, G);
        int op = __shfl_xor_sync(gmask, minP, o, G), os = __shfl_xor_sync(gmask, minSeq, o, G);
        if (op >= 0 && (oa < minAlpha || (oa == minAlpha && os > minSeq))) { minAlpha = oa; minP = op; minSeq = os; }
      }
      if (minP < 0 || 1.0f - 10.0f * B2_EPS < minAlpha) break;   // group-uniform
      int ea, ek, eb; decode(minP, ea, ek, eb);   // the event's contact: static body ek, agent eb
      const bool mine = eb == g;
      if (mine) cvalid &= ~(1u << ek);
      gsync();
      int r = 0;
      TOIPROF(long long tpe = clock64();)
      if (lead) {
        RARE_BEGIN();
        if ((MSV_INLINE_MASK >> 1) & 1) r = toi_event(minP, minAlpha, dt, prevP);
        else { Env c_(*this); r = c_.toi_event(minP, minAlpha, dt, prevP); take(c_); }
        if (r & 1) prevP = minP;
        RARE_END(1);
      }
      gsync();
      r = bc(r);
      TOIPROF(tp_ev += clock64() - tpe; if (r & 1) tp_ran++; else tp_not++; if (r & 2) tp_same++;)
      share_bits();
      if (mine) {                              // toiCount of the event's contact (saturating at 15 > b2_maxSubSteps)
        const unsigned long long c4 = (evcnt >> (4 * ek)) & 15ull;
        if (c4 < 15ull) evcnt += 1ull << (4 * ek);
      }
      if (!(r & 1)) continue;
      if (mine) {
        if (r & 2) {
          // identical repeat: every further event on this contact would repeat verbatim -> jump its toiCount past
          // b2_maxSubSteps.  The agent's state is exactly what it was after the previous event, so the TOIs of its
          // other contacts, computed from that state, are still the ones SolveTOI would recompute: keep them.
          const unsigned long long c4 = (evcnt >> (4 * ek)) & 15ull;
          if (c4 <= (unsigned long long)C.toi_max_count) evcnt = (evcnt & ~(15ull << (4 * ek))) | ((unsigned long long)(C.toi_max_count + 1) << (4 * ek));
        } else cvalid = 0u;                    // "Invalidate all contact TOIs on this displaced body"
      }
    }
    gsync();
    TOIPROF(if (lead) { unsigned long long tot = (unsigned long long)(clock64() - tp0); unsigned long long old = atomicMax(&g_toi[0], tot);
      if (tot > old) { g_toi[1] = tp_it; g_toi[2] = tp_ran; g_toi[3] = tp_not; g_toi[4] = tp_same; g_toi[5] = (unsigned long long)tp_ev; g_toi[6] = tot - (unsigned long long)tp_ev; g_toi[7] = tp_calls; g_toi[8] = (unsigned long long)e; } })
  }

  // ======================================================================
  //                      SEMANTICS (pre_step / post_step)
  // ======================================================================
  // agents/DynamicMotors.pre_step (sim:407-424)                      [all lanes]
  // Returns the group's action flags: bit i attack, bit 8+i use, bit 16+i give of agent i.
  __device__ __forceinline__ unsigned pre_motors(const uint8_t* actions, bool real) {
    unsigned flags = 0;
    for (int i = g; i < C.A; i += G) {
      int a0 = 1, a1 = 1, a2 = 1;            // padding envs (N rounded up to the block size) get the no-op action
      if (real) {
        const uint8_t* a = actions + ((size_t)e * C.A + i) * 6;
        a0 = min((int)a[0], 2); a1 = min((int)a[1], 2); a2 = min((int)a[2], 2);   // env:80 asserts the range; never index past the tables
        flags |= (a[3] ? 1u : 0u) << i | (a[4] ? 1u : 0u) << (8 + i) | (a[5] ? 1u : 0u) << (16 + i);
      }
      if (!alive(i)) continue;
      float s, c; rot_set(AG(F_A, i), s, c);
      AG(F_QS, i) = s; AG(F_QC, i) = c;
      float par = C.imp_par[a0], nor = C.imp_nor[a1];
      float ix = c * par + (-s) * nor, iy = s * par + c * nor;
      wake(i);
      AG(F_VX, i) += C.inv_mass * ix; AG(F_VY, i) += C.inv_mass * iy;
      AG(F_W, i) += C.inv_I * C.imp_ang[a2];
    }
    return or32(flags);
  }
  // [leader] pending drops, UseLast, GiveLast
  DEV void pre_use_give(unsigned act) {
    LI(L_USEHEAL) = 0; LI(L_USEBOX) = 0; LI(L_NEWBOX) = 0;
    bool any = LI(L_NP) > 0;                       // nothing to do unless a drop is pending or an agent with items uses/gives
#pragma unroll
    for (int i = 0; i < AC; ++i) if (i < C.A && (((act >> (8 + i)) | (act >> (16 + i))) & 1u) && (LI(L_INV + (i)) & 7) != 0 && alive(i)) any = true;
    if (any) { RARE_BEGIN(); MSV_COLDK(3, pre_use_give_body(act)); RARE_END(5); }
  }
  COLD3 void pre_use_give_body(unsigned act) {
    // boxes/Object.pre_step (sem:853-856, 902-905): pending drops become items
    for (int q = 0; q < LI(L_NP); ++q) {
      float4 p0 = S.pend0[q * N + e];
      add_item(p0.x, p0.y, p0.z, p0.w, S.pend1[q * N + e]);
    }
    LI(L_NP) = 0;
    // agents/UseLast.pre_step (sem:300-309) -> Inventory.use (sem:206-213)
#pragma unroll
    for (int i = 0; i < AC; ++i) {
      if (i >= C.A || !alive(i) || !((act >> (8 + i)) & 1u) || inv_n(i) == 0) continue;
      float4 pl; int kind = inv_pop(i, pl);
      if (kind == MSV_ITEM_HEAL) { LI(L_USEHEAL)++; agent_change_health(i, C.healing, MSV_CAUSE_NONE); }  // sem:646-649
      else {  // ObjectItem.use (sem:830-836, 876-884)
        LI(L_USEBOX)++;
        if (nb >= BC) { LI(L_OVERFLOW)++; continue; }
        float L = C.box_item_offset;
        float qs = AG(F_QS, i), qc = AG(F_QC, i);
        f2 off = mk2(qc * L + (-qs) * 0.0f, qs * L + qc * 0.0f);
        float x = AG(F_CX, i) + off.x, y = AG(F_CY, i) + off.y;
        int reh = __float_as_int(pl.w) & 1;
        const float4 nb0 = make_float4(x, y, pl.x, pl.y);
        const int4 nb1 = make_int4(0, reh << 1, MSV_CAUSE_NONE, C.box_ownership ? __float_as_int(pl.z) : MSV_CAUSE_NONE);
        S.box0[nb * N + e] = nb0; S.box1[nb * N + e] = nb1;
        S.boxseq[nb * N + e] = LI(L_BODYSEQ)++;
        put_box(nb, nb0, nb1);                       // (not read back from global memory)
        for (int j = 0; j < C.A; ++j) { int p = p_ab(j, nb); clrb(ex, p); clrb(tc, p); clrb(en, p); }
        nb++; LI(L_NEWBOX) = 1; LI(L_NEWFIX) = 1;
      }
    }
    // agents/GiveLast.pre_step (sem:335-370): taker = nearest body of any kind
#pragma unroll
    for (int i = 0; i < AC; ++i) {
      if (i >= C.A || !alive(i) || !((act >> (16 + i)) & 1u) || inv_n(i) == 0) continue;
      f2 me = apos(i); float r2 = C.give_r * C.give_r;
      float minDist = INFINITY; int tkind = KIND_NONE, tidx = -1;
      auto consider = [&](f2 o, int kind, int idx) {
        f2 d = vsub(o, me);
        if (!(vdot(d, d) <= r2)) return;                 // b2CircleShape::TestPoint
        f2 dd = vsub(me, o);
        float dist = sqrtf(dd.x * dd.x + dd.y * dd.y);
        if (dist < minDist) { minDist = dist; tkind = kind; tidx = idx; }
      };
      for (int k = 0; k < nb; ++k) consider(mk2(BX(G_X, k), BX(G_Y, k)), KIND_BOX, k);
      for (int k = 0; k < ni; ++k) { float4 it = S.item0[k * N + e]; consider(mk2(it.x, it.y), KIND_ITEM, k); }
      for (int k = 0; k < nh; ++k) { float2 h = S.heal[k * N + e]; consider(mk2(h.x, h.y), KIND_HEAL, k); }
      for (int k = 0; k < 4; ++k) consider(mk2(C.walls[k].px, C.walls[k].py), KIND_WALL, k);
      for (int j = 0; j < C.A; ++j) if (j != i && alive(j)) consider(apos(j), KIND_AGENT, j);
      if (tkind != KIND_AGENT) continue;                               // sem:196-198
      if (C.teams && team_of(tidx) != team_of(i)) continue;            // strangers sem:344-349
      float4 pl = make_float4(0.f, 0.f, 0.f, 0.f); int kind = inv_pop(i, pl);
      if (inv_n(tidx) + 1 <= C.inv_slots) {
        inv_push(tidx, kind, pl);
      }                                                                // else lost (Q6)
    }
  }
  // agents/Melee.pre_step (sem:584-617) / ContinuousMelee (sem:531-554).  The
  // rays only depend on geometry (boxes placed above included), which the
  // health changes do not alter: every lane casts its agents' rays, then the
  // leader applies the hits in agent order.                          [all lanes]
  __device__ __forceinline__ void pre_melee(unsigned act) {
    unsigned raymask = 0;
    if (lead) {
#pragma unroll
      for (int i = 0; i < AC; ++i) {
        if (i >= C.A || !alive(i)) continue;
        bool on_cd = C.melee_cooldown >= 0 && LI(L_COOLDOWN + (i)) > 0;
        if (((act >> i) & 1u) && !on_cd) raymask |= 1u << i;
      }
    }
    raymask = bc(raymask);
    if (raymask) {                             // group-uniform
      int res[AC];
#pragma unroll
      for (int s = 0; s < SLOTS; ++s) {
        const int i = s * G + g;
        int r = 0;
        if ((raymask >> i) & 1u) {
          f2 me = apos(i);
          float L = C.melee_range, qs = AG(F_QS, i), qc = AG(F_QC, i);
          f2 hand = mk2(qc * L + (-qs) * 0.0f, qs * L + qc * 0.0f);
          int tidx; float frac;
          int kind = raycast(me, vadd(me, hand), i, tidx, frac);
          r = kind | ((tidx & 255) << 8);
        }
#pragma unroll
        for (int j = 0; j < G; ++j) res[s * G + j] = from(r, j);
      }
      if (lead) {
#pragma unroll
        for (int i = 0; i < AC; ++i) {
          if (!((raymask >> i) & 1u)) continue;
          int kind = res[i] & 255, tidx = (res[i] >> 8) & 255;
          if (kind == KIND_NONE) continue;
          int cz = C.teams ? MSV_CAUSE_TEAM0 + team_of(i) : i;
          if (kind == KIND_AGENT) agent_change_health(tidx, -C.melee_damage, cz);
          else if (kind == KIND_BOX) box_change_health(tidx, -C.melee_damage, cz);
          if (C.melee_cooldown >= 0) LI(L_COOLDOWN + (i)) = C.melee_cooldown;
        }
      }
    }
    if (lead && C.melee_cooldown >= 0) {
#pragma unroll
      for (int i = 0; i < AC; ++i) if (LI(L_COOLDOWN + (i)) > 0) LI(L_COOLDOWN + (i))--;
    }
  }

  __device__ __noinline__ double philox_uniform(uint32_t step, uint32_t stream, uint32_t k) {
    uint32_t o[4];
    philox4x32(C.env_offset + (uint32_t)e, (uint32_t)LI(L_EPISODE), step, (stream << 16) | (k >> 1), C.seed_lo, C.seed_hi, o);
    uint32_t a = o[(k & 1) * 2], b = o[(k & 1) * 2 + 1];
    return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) / 9007199254740992.0;
  }

  // Cameras._update_seen (sim:336-354), agent targets (the only ones the
  // omniscient observation reads, env:692-703)
  DEV bool in_cone(f2 pl) {                          // b2PolygonShape::TestPoint(vision cone)
    bool inside = true;
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      float d = vdot(mk2(C.cone_n[v][0], C.cone_n[v][1]), vsub(pl, mk2(C.cone_v[v][0], C.cone_v[v][1])));
      if (d > 0.0f) inside = false;
    }
    return inside;
  }
  // position of camera target t: [0,AC) agents, then BC boxes, BC box items, HC heals
  DEV f2 target_pos(int t) {
    if (t < AC) return apos(t);
    t -= AC;
    if (t < BC) return mk2(BX(G_X, t), BX(G_Y, t));
    t -= BC;
    if (t < BC) return mk2(ITP(0, t), ITP(1, t));
    t -= BC;
    return mk2(HLP(0, t), HLP(1, t));
  }
  // every lane is the camera of its own agents                      [all lanes]
  DEV void cameras() {
    gsync();
    const bool all_bodies = !C.omniscient;            // env:706-739 read the full seen-lists
    unsigned saL[SLOTS], sxL[SLOTS];
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
      const int i = s * G + g;
      unsigned sa = 0, sx = 0;
      if (i < C.A && alive(i)) {
        // pass 1: which targets have their centre inside the cone
        f2 me = apos(i); float sn, cs; rot_set(AG(F_A, i), sn, cs);
        unsigned long long m = 0ull;
        for (int j = 0; j < C.A; ++j)
          if (j != i && alive(j) && in_cone(qmulT(sn, cs, vsub(apos(j), me)))) m |= 1ull << j;
        if (all_bodies) {
          for (int k = 0; k < nb; ++k) if (in_cone(qmulT(sn, cs, vsub(target_pos(AC + k), me)))) m |= 1ull << (AC + k);
          for (int k = 0; k < ni; ++k) if (in_cone(qmulT(sn, cs, vsub(target_pos(AC + BC + k), me)))) m |= 1ull << (AC + BC + k);
          for (int k = 0; k < nh; ++k) if (in_cone(qmulT(sn, cs, vsub(target_pos(AC + 2 * BC + k), me)))) m |= 1ull << (AC + 2 * BC + k);
        }
        // pass 2: one line-of-sight ray per in-cone target
        while (m) {
          int t = __ffsll((long long)m) - 1; m &= m - 1;
          f2 o = target_pos(t);
          f2 d = vsub(o, me);
          f2 end = mk2(me.x + C.cam_k1 * d.x, me.y + C.cam_k1 * d.y);
          int idx; float fr;
          int kind = raycast(me, end, i, idx, fr);
          if (t < AC) { if (kind == KIND_AGENT && idx == t) sa |= 1u << t; }
          else if (t < AC + BC) { if (kind == KIND_BOX && idx == t - AC) sx |= 1u << (16 + t - AC); }
          else if (t < AC + 2 * BC) { if (kind == KIND_ITEM && idx == t - AC - BC) sx |= 1u << (24 + t - AC - BC); }
          else { if (kind == KIND_HEAL && idx == t - AC - 2 * BC) sx |= 1u << (t - AC - 2 * BC); }
        }
      }
      saL[s] = sa; sxL[s] = sx;
    }
    // rows of Cameras.seen are in the order of the bodies alive NOW (before this step's deaths)
    unsigned saA[AC], sxA[AC];
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
#pragma unroll
      for (int j = 0; j < G; ++j) { saA[s * G + j] = from(saL[s], j); sxA[s * G + j] = from(sxL[s], j); }
    }
    if (lead) {
      LU(L_PREALIVE) = 0; int row = 0;
#pragma unroll
      for (int i = 0; i < AC; ++i) { LU(L_SEENA + (i)) = 0; LU(L_SEENX + (i)) = 0; }
#pragma unroll
      for (int i = 0; i < AC; ++i) {
        if (i >= C.A || !alive(i)) continue;
        LU(L_PREALIVE) |= 1u << i;
        LU(L_SEENA + row) = saA[i]; LU(L_SEENX + row) = sxA[i];
        row++;
      }
    }
  }
  // a floor item / heal left its list after the cameras ran: compact the seen bits
  DEV void seen_remove(int first_bit, int width, int k) {
#pragma unroll
    for (int r = 0; r < AC; ++r) {
      unsigned field = (LU(L_SEENX + (r)) >> first_bit) & ((1u << width) - 1u);
      unsigned lowm = (1u << k) - 1u;
      field = (field & lowm) | ((field >> (k + 1)) << k);
      LU(L_SEENX + (r)) = (LU(L_SEENX + (r)) & ~(((1u << width) - 1u) << first_bit)) | (field << first_bit);
    }
  }


  // [leader]
  __device__ __forceinline__ void post_step_boxes() {
    // boxes/Health.post_step (sem:429-435) + Object.pre_despawn (sem:858-861, 911-912)
    // (the health words of all boxes are fetched together: one memory latency instead of one per box)
    int4 b1s[BC];
#pragma unroll
    for (int j = 0; j < BC; ++j) if (j < nb) b1s[j] = S.box1[j * N + e];
    const int nb0 = nb; int removed = 0;
#pragma unroll
    for (int j = 0; j < BC; ++j) {
      if (j >= nb0) continue;
      const int k = j - removed;                  // current list position of the box that was at j
      int4 b1 = b1s[j];
      if (!(b1.y & 1)) { b1.y |= 1; b1.x = C.box_health; S.box1[k * N + e] = b1; }
      if (b1.x <= 0) {
        if (LI(L_NP) < BC) {
          S.pend0[LI(L_NP) * N + e] = make_float4(BX(G_X, k), BX(G_Y, k), BX(G_HX, k), BX(G_HY, k));
          S.pend1[LI(L_NP) * N + e] = C.box_ownership ? b1.z : MSV_CAUSE_NONE;
          LI(L_NP)++;
        } else LI(L_OVERFLOW)++;
        { RARE_BEGIN(); MSV_COLDK(3, remove_box(k)); RARE_END(7); }
        removed++;
      }
    }
  }
  // agents/Cameras.post_step (sim:333-334) runs between the two halves
  // [leader] agents/Health.post_step -> despawn(dead) (sem:429-448)
  COLD3 void handle_deaths() {
    int total = 0;
    for (int i = 0; i < C.A; ++i) if ((LU(L_DMASK) >> i) & 1u) total += inv_n(i);
    int top = total;
    for (int i = 0; i < C.A; ++i) {         // DeathDrop.pre_despawn (sem:387-396)
      if (!((LU(L_DMASK) >> i) & 1u)) continue;
      f2 me = apos(i);
      int n = inv_n(i);
      for (int j = 0; j < n; ++j) {
        double ang = 2 * 3.141592653589793 * philox_uniform((uint32_t)LI(L_STEPS), STREAM_DEATH, (uint32_t)(--top));
        f2 off = from_polar(C.drop_radius, (float)ang);
        float x = me.x + off.x, y = me.y + off.y;
        int kind = inv_kind(i, j);
        if (kind == MSV_ITEM_HEAL) add_heal(x, y);
        else { float4 pl = S.ainv[(i * 4 + j) * N + e]; add_item(x, y, pl.x, pl.y, __float_as_int(pl.z)); }
      }
      LI(L_INV + (i)) = 0;
    }
    for (int i = 0; i < C.A; ++i) if ((LU(L_DMASK) >> i) & 1u) LI(L_KCAUSE + (LI(L_NKILLS)++)) = LI(L_CAUSE + (i));  // TrackKills sem:628-629
    for (int i = 0; i < C.A; ++i) if ((LU(L_DMASK) >> i) & 1u) kill_agent(i);
  }
  // pairs that involve agent i (compile-time masks)
  DEV static constexpr unsigned long long pairs_of(int i, int w) {
    unsigned long long m = 0ull;
    for (int j = 0; j < AC; ++j) if (j != i) { const int p = i < j ? j * (j - 1) / 2 + i : i * (i - 1) / 2 + j; if ((p >> 6) == w) m |= 1ull << (p & 63); }
    for (int k = 0; k < BC + 4; ++k) { const int p = k < BC ? NAA + i * BC + k : NAA + AC * BC + i * 4 + (k - BC); if ((p >> 6) == w) m |= 1ull << (p & 63); }
    return m;
  }
  // [leader] handle_deaths() for agents that carry nothing: TrackKills (sem:628-629) in index order, then
  // b2World::DestroyBody for each (touching agent-agent contacts wake the partner), all with static pair masks
  DEV void kill_agents_empty(unsigned dm) {
#pragma unroll
    for (int i = 0; i < AC; ++i) if ((dm >> i) & 1u) LI(L_KCAUSE + (LI(L_NKILLS)++)) = LI(L_CAUSE + (i));
#pragma unroll
    for (int i = 0; i < AC; ++i) {
      if (!((dm >> i) & 1u)) continue;
#pragma unroll
      for (int j = 0; j < AC; ++j) {
        if (j == i) continue;
        const int p = i < j ? j * (j - 1) / 2 + i : i * (i - 1) / 2 + j;     // p_aa, static
        if (((ex[0] & tc[0]) >> p) & 1ull) wake(j);
      }
#pragma unroll
      for (int w = 0; w < PW; ++w) { const unsigned long long m = ~pairs_of(i, w); ex[w] &= m; tc[w] &= m; en[w] &= m; }
      AGF(i) = 0;
    }
  }
  // [leader] agents/AutoPickup.post_step (sem:278-283) for agent i: bodies in creation order
  COLD3 void pickup_agent(int i) {
    const float r2 = C.pickup_r * C.pickup_r;
    f2 me = apos(i);
    int lastSeq = -1;
    for (;;) {
      int bestSeq = 0x7FFFFFFF, bkind = KIND_NONE, bidx = -1;
      for (int k = 0; k < ni; ++k) {
        float4 it = S.item0[k * N + e]; f2 d = vsub(mk2(it.x, it.y), me);
        if (!(vdot(d, d) <= r2)) continue;
        int sq = S.item1[k * N + e].y;
        if (sq > lastSeq && sq < bestSeq) { bestSeq = sq; bkind = KIND_ITEM; bidx = k; }
      }
      for (int k = 0; k < nh; ++k) {
        float2 h = S.heal[k * N + e]; f2 d = vsub(mk2(h.x, h.y), me);
        if (!(vdot(d, d) <= r2)) continue;
        int sq = S.healseq[k * N + e];
        if (sq > lastSeq && sq < bestSeq) { bestSeq = sq; bkind = KIND_HEAL; bidx = k; }
      }
      if (bkind == KIND_NONE) break;
      lastSeq = bestSeq;
      if (inv_n(i) + 1 > C.inv_slots) continue;  // sem:184-185
      if (bkind == KIND_HEAL) { inv_push(i, MSV_ITEM_HEAL, make_float4(0.f, 0.f, 0.f, 0.f)); remove_heal(bidx); seen_remove(0, 16, bidx); }
      else {
        float4 it = S.item0[bidx * N + e]; int2 i1 = S.item1[bidx * N + e];
        inv_push(i, MSV_ITEM_BOX, make_float4(it.z, it.w, __int_as_float(i1.x), __int_as_float(1)));
        remove_item(bidx); seen_remove(24, 8, bidx);
      }
    }
  }
  // [all lanes] the post_step hooks after the cameras.  Every lane pre-checks
  // whether anything lies within pickup range of its own agents (removals by
  // earlier agents can only shrink that set), the leader runs the exact
  // sequential pickups for those agents only.
  __device__ __forceinline__ void post_step_rest() {
    int dflag = 0;
    if (lead) {
      LU(L_DMASK) = 0; LI(L_NKILLS) = 0;
#pragma unroll
      for (int i = 0; i < AC; ++i) if (i < C.A && alive(i) && LI(L_HEALTH + (i)) <= 0) LU(L_DMASK) |= 1u << i;
      if (LU(L_DMASK)) {
        const unsigned dm = LU(L_DMASK);
        int carried = 0;
#pragma unroll
        for (int i = 0; i < AC; ++i) if ((dm >> i) & 1u) carried += LI(L_INV + (i)) & 7;
        if (carried == 0) kill_agents_empty(dm);      // nothing to drop (the usual case): TrackKills + DestroyBody only
        else { RARE_BEGIN(); MSV_COLDK(3, handle_deaths()); RARE_END(3); }
        dflag = 1;
      }
    }
    dflag = bc(dflag);
    if (dflag) { gsync(); share_counts(); }   // drops changed the lists, deaths the flags
    unsigned near = 0;
    {
      const float r2 = C.pickup_r * C.pickup_r;
      for (int i = g; i < C.A; i += G) {
        if (!alive(i)) continue;
        f2 me = apos(i); bool any = false;
        for (int k = 0; k < ni; ++k) { f2 d = vsub(mk2(ITP(0, k), ITP(1, k)), me); if (vdot(d, d) <= r2) any = true; }
        for (int k = 0; k < nh; ++k) { f2 d = vsub(mk2(HLP(0, k), HLP(1, k)), me); if (vdot(d, d) <= r2) any = true; }
        if (any) near |= 1u << i;
      }
    }
    near = or32(near);
    if (!lead) return;
    for (int i = 0; i < C.A; ++i) if ((near >> i) & 1u) { RARE_BEGIN(); MSV_COLDK(3, pickup_agent(i)); RARE_END(4); }
    // agents/SafeZone.post_step (sem:758-768) + tick (sem:776-811)
    for (int i = 0; i < C.A; ++i) {
      if (!alive(i)) continue;
      float dx = AG(F_CX, i) - LF(L_ZX), dy = AG(F_CY, i) - LF(L_ZY);
      bool inside = dx * dx + dy * dy <= LF(L_ZR) * LF(L_ZR);
      if (LI(L_ZEND) || !inside) agent_change_health(i, -C.zone_damage, MSV_CAUSE_ZONE);
    }
    if (LI(L_ZTCOOL) == 0) {
      if (!LI(L_ZEND)) {
        LI(L_ZTSHRINK) -= 1;
        if (LI(L_ZTSHRINK) > 0) {
          double t = (double)LI(L_ZTSHRINK) / C.zone_cooldown;
          double r1 = C.zone_radiuses[LI(L_ZPHASE)], r2 = C.zone_radiuses[LI(L_ZPHASE) + 1];
          LF(L_ZR) = (float)(t * r1 + (1 - t) * r2);
          float t1 = (float)t, t2 = (float)(1 - t);
          float2 c1 = S.zonec[LI(L_ZPHASE) * N + e], c2 = S.zonec[(LI(L_ZPHASE) + 1) * N + e];
          LF(L_ZX) = t1 * c1.x + t2 * c2.x; LF(L_ZY) = t1 * c1.y + t2 * c2.y;
        } else {
          LI(L_ZTCOOL) = C.zone_cooldown; LI(L_ZPHASE) += 1;
          LF(L_ZR) = C.zone_r32[LI(L_ZPHASE)];
          float2 cc = S.zonec[LI(L_ZPHASE) * N + e]; LF(L_ZX) = cc.x; LF(L_ZY) = cc.y;
          if (LI(L_ZPHASE) == C.zone_phases - 1) LI(L_ZEND) = 1;
        }
      }
    } else {
      LI(L_ZTCOOL) -= 1;
      if (LI(L_ZTCOOL) <= 0) LI(L_ZTSHRINK) = C.zone_cooldown;
    }
  }

  // ======================================================================
  //                 OBSERVATIONS / REWARDS / DONE / STATS
  // ======================================================================
  // others_mask (env:692-703) as bits: bit (i*AC + j) set <=> observer i sees
  // agent j.  Q1: Cameras.seen is looked up by the POST-death list position.
  // The observation tensors themselves are written by k_obs2 (msv_kernels.cu).
  // [leader]
  DEV void store_obm() {
    unsigned long long bits = 0ull;
    unsigned am = 0;                           // agents alive now (after this step's deaths)
    for (int i = 0; i < C.A; ++i) if (alive(i)) am |= 1u << i;
    int r = 0;
    for (int i = 0; i < C.A; ++i) {
      if (!((am >> i) & 1u)) continue;
      const unsigned sr = LU(L_SEENA + r);
      r++;
      bits |= (unsigned long long)(sr & am & ~(1u << i)) << (i * AC);
    }
    S.obm[e] = bits;
    if (!C.omniscient) {   // env:706-739: zip(agents.bodies, cameras.seen) -> same Q1 row remap
      int r2 = 0;
      for (int i = 0; i < C.A; ++i) {
        unsigned sx = 0;
        if (alive(i)) {
          sx = LU(L_SEENX + r2);
          r2++;
        }
        S.omask[i * N + e] = sx;
      }
    }
  }

  DEV bool team_alive(int t) {
    int split = C.A / 2; bool any = false;
    for (int i = (t ? split : 0); i < (t ? C.A : split); ++i) any |= alive(i);
    return any;
  }

  // compute_rewards (env:757-803), is_done (env:810-831), _update_stats (env:483-508)   [leader]
  // (register arrays are only indexed by unrolled loop counters)
  DEV bool rewards_done(DevOut& O) {
    const int A = C.A, split = A / 2;
    float rew[AC]; int lk[AC];
#pragma unroll
    for (int i = 0; i < AC; ++i) { rew[i] = 0.0f; lk[i] = 0; }
    const bool ta0 = team_alive(0), ta1 = team_alive(1);
    if (!C.teams) {
#pragma unroll
      for (int i = 0; i < AC; ++i) if (i < A) rew[i] += alive(i) ? C.r_alive : C.r_dead;
      for (int k = 0; k < LI(L_NKILLS); ++k) {
        int killer = LI(L_KCAUSE + (k));
        if (killer >= 0 && killer < A && alive(killer)) {
#pragma unroll
          for (int i = 0; i < AC; ++i) if (i == killer) { rew[i] += C.r_kill; lk[i]++; }
        }
      }
      if (LU(L_DMASK)) {
#pragma unroll
        for (int i = 0; i < AC; ++i) if ((LU(L_DMASK) >> i) & 1u) rew[i] += C.r_death;
      }
    } else {
#pragma unroll
      for (int i = 0; i < AC; ++i) if (i < A) rew[i] += (i < split ? ta0 : ta1) ? C.r_alive : C.r_dead;
      for (int k = 0; k < LI(L_NKILLS); ++k) {
        int cz = LI(L_KCAUSE + (k));
        if (cz != MSV_CAUSE_TEAM0 && cz != MSV_CAUSE_TEAM0 + 1) continue;
        int t = cz - MSV_CAUSE_TEAM0;
#pragma unroll
        for (int i = 0; i < AC; ++i) if (i < A && (i < split ? 0 : 1) == t) rew[i] += C.r_kill;
#pragma unroll
        for (int i = 0; i < 2; ++i) if (i == t) lk[i]++;
      }
      if (LU(L_DMASK)) {
        for (int d = 0; d < A; ++d) {         // deaths in index order
          if (!((LU(L_DMASK) >> d) & 1u)) continue;
          int t = team_of(d);
#pragma unroll
          for (int i = 0; i < AC; ++i) if (i < A && (i < split ? 0 : 1) == t) rew[i] += C.r_death;
        }
      }
    }
    int n_alive = 0;
    if (C.teams) n_alive = (int)ta0 + (int)ta1;
    else for (int i = 0; i < A; ++i) n_alive += alive(i);
    bool done = C.gameover_mode == MSV_GAMEOVER_ALLDEAD ? n_alive == 0 : n_alive <= 1;
    LI(L_STEPS) += 1;
    if (!C.teams) {
#pragma unroll
      for (int i = 0; i < AC; ++i) if (i < A) LF(L_SREW + (i)) += rew[i];
    } else {
      LF(L_SREW + (0)) += rew[0];
      float rs = 0.0f;
#pragma unroll
      for (int i = 0; i < AC; ++i) if (i == split) rs = rew[i];
      LF(L_SREW + (1)) += rs;
    }
#pragma unroll
    for (int i = 0; i < AC; ++i) if (i < (C.teams ? 2 : A)) LI(L_SKILLS + (i)) += lk[i];
    LI(L_STSTEPS) += 1; LI(L_STHEALS) += LI(L_USEHEAL); LI(L_STBOXES) += LI(L_USEBOX);
#pragma unroll
    for (int i = 0; i < AC; ++i) if (i < A) { O.rewards[(size_t)e * A + i] = rew[i]; LF(L_EPRET + (i)) += rew[i]; }
    O.dones[e] = done ? 1 : 0;
    if (done) {   // per-env episode statistics of the episode that just ended (rows valid where dones)
#pragma unroll
      for (int i = 0; i < AC; ++i) if (i < A) O.episode_return[(size_t)e * A + i] = LF(L_EPRET + (i));
      O.episode_length[e] = LI(L_STEPS);
    }
    if (C.battle_royale) {   // BattleRoyale.post_step (sem:41-46): runs last, on the post-death body list
      int na = 0;
      for (int i = 0; i < A; ++i) na += alive(i);
      O.br_over[e] = na <= 1 ? 1 : 0;
      for (int i = 0; i < A; ++i) O.br_results[(size_t)e * A + i] = (na <= 1 && alive(i)) ? 1 : 0;   // .results only exists once over
    }
    return done;
  }

  // ======================================================================
  //                               RESET
  // ======================================================================
  // BaseEnv.reset (env:59-74): SpawnGrid (sem:59-79), ResetSpawns (sem:82-94),
  // RandomizeBoxShapes (sem:97-120), ThickRoomWalls, SafeZone.post_reset
  // (sem:739-756).  The numpy Generator is replaced by counter-based
  // Philox4x32-10 keyed by (seed, global env id, episode).          [leader]
  COLD4 void reset() {
    LI(L_EPISODE) += 1; LI(L_STEPS) = 0;
    // the episode's random draws: the record k_spare prepared, or (no record for this episode yet) drawn now.
    // It is staged in the dead touching-contact list of the environment's shared-memory column.
    float* rec = &msv_sm[sb + W_TC];
    static_assert(K_COUNT * MAXC >= MSV_SPARE_W, "scratch too small for a reset record");
    if (S.spare_ep[e] == LI(L_EPISODE)) {
      const float4* src = reinterpret_cast<const float4*>(S.spare + (size_t)e * MSV_SPARE_W);
      float4 v[MSV_SPARE_W / 4];
#pragma unroll
      for (int q = 0; q < MSV_SPARE_W / 4; ++q) v[q] = src[q];         // one memory latency
#pragma unroll
      for (int q = 0; q < MSV_SPARE_W / 4; ++q) { rec[4 * q] = v[q].x; rec[4 * q + 1] = v[q].y; rec[4 * q + 2] = v[q].z; rec[4 * q + 3] = v[q].w; }
    } else draw_reset(C, C.env_offset + (uint32_t)e, (uint32_t)LI(L_EPISODE), rec);
    LI(L_BODYSEQ) = 0; LI(L_CONTACTSEQ) = 0; LI(L_FIRST) = 1; LI(L_NEWFIX) = 1;
    nb = 0; ni = 0; nh = 0; LI(L_NP) = 0;
#pragma unroll
    for (int w = 0; w < PW; ++w) { ex[w] = 0ull; tc[w] = 0ull; en[w] = 0ull; }
#pragma unroll 1
    for (int b = 0; b < C.B0; ++b) {
      const float4 nb0 = make_float4(rec[MSV_SP_BOX + 4 * b], rec[MSV_SP_BOX + 4 * b + 1], rec[MSV_SP_BOX + 4 * b + 2], rec[MSV_SP_BOX + 4 * b + 3]);
      const int4 nb1 = make_int4(C.box_health, 1, MSV_CAUSE_NONE, MSV_CAUSE_NONE);
      S.box0[b * N + e] = nb0; S.box1[b * N + e] = nb1;
      S.boxseq[b * N + e] = LI(L_BODYSEQ)++;
      put_box(b, nb0, nb1);                          // (not read back from global memory)
      nb++;
    }
#pragma unroll 1
    for (int h = 0; h < C.H0; ++h) {
      const float x = rec[MSV_SP_HEAL + 2 * h], y = rec[MSV_SP_HEAL + 2 * h + 1];
      S.heal[h * N + e] = make_float2(x, y); HLP(0, h) = x; HLP(1, h) = y;
      S.healseq[h * N + e] = LI(L_BODYSEQ)++;
      nh++;
    }
    LI(L_BODYSEQ) += 4;  // walls
#pragma unroll 1
    for (int i = 0; i < AC; ++i) {
      if (i < C.A) {
        const float x = rec[MSV_SP_AGENT + 2 * i], y = rec[MSV_SP_AGENT + 2 * i + 1], r = C.agent_r;
        AG(F_CX, i) = x; AG(F_CY, i) = y; AG(F_A, i) = 0.0f; AG(F_VX, i) = 0.0f; AG(F_VY, i) = 0.0f; AG(F_W, i) = 0.0f;
        AG(F_C0X, i) = x; AG(F_C0Y, i) = y; AG(F_A0, i) = 0.0f; AG(F_ALPHA0, i) = 0.0f; AG(F_SLEEP, i) = 0.0f;
        AG(F_FAT0, i) = (x - r) - B2_AABB_EXT; AG(F_FAT1, i) = (y - r) - B2_AABB_EXT;
        AG(F_FAT2, i) = (x + r) + B2_AABB_EXT; AG(F_FAT3, i) = (y + r) + B2_AABB_EXT;
        AGF(i) = FL_ALIVE | FL_AWAKE;
        LI(L_HEALTH + (i)) = C.health; LI(L_BODYSEQ)++;
      } else { AGF(i) = 0; LI(L_HEALTH + (i)) = 0; }
      LI(L_CAUSE + (i)) = MSV_CAUSE_NONE; LI(L_COOLDOWN + (i)) = 0; LI(L_INV + (i)) = 0;
      LF(L_EPRET + (i)) = 0.0f;
    }
#pragma unroll 1
    for (int z = 0; z < C.n_zones; ++z) S.zonec[z * N + e] = make_float2(rec[MSV_SP_ZONE + 2 * z], rec[MSV_SP_ZONE + 2 * z + 1]);
    LI(L_ZTCOOL) = C.zone_cooldown; LI(L_ZTSHRINK) = 0; LI(L_ZPHASE) = 0; LI(L_ZEND) = 0;
    LF(L_ZR) = C.zone_r32[0];
    LF(L_ZX) = rec[MSV_SP_ZONE]; LF(L_ZY) = rec[MSV_SP_ZONE + 1];
    LU(L_DMASK) = 0; LI(L_NKILLS) = 0; LI(L_USEHEAL) = 0; LI(L_USEBOX) = 0;
  }
  // ImmunityPhase (sem:652-674): Health.immune is True from reset until max(cooldown, 1) steps have run  [leader]
  DEV void store_immune(DevOut& O) {
    if (C.immunity_cooldown < 0) return;
    const int cd = C.immunity_cooldown < 1 ? 1 : C.immunity_cooldown;
    O.immune[e] = LI(L_STEPS) < cd ? 1 : 0;
  }
};
