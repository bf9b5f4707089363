// msv_render.cu -- top-down RGB picture of environments straight from the SoA state in HBM (msv_render).
//
// The picture (tests/render_reference.py restates it in numpy float32 and must match every byte):
//   * uint8[H][W][3], row 0 at the top, +y up.  Viewport: a square of half-width V = (float)(F/2 + F/100)
//     (F = floor_size) centred on the origin, pixel size s = 2V / min(W, H); the centre of pixel (column i,
//     row j) is x = ((float)(2i - W + 1) * 0.5f) * s, y = ((float)(H - 1 - 2j) * 0.5f) * s.
//   * Layers, later on top, each a predicate on the pixel centre: background; floor (|x|, |y| <= F/2);
//     floor outside the current safe zone; the current zone's ring, then the next zone's; walls; heals;
//     box items (their sensor circle); boxes; living agents (index order); their heading ticks; with
//     MSV_RENDER_LIDAR their rays, cut at the current lidar_frac.
//   * Only float32 + - * / and comparisons (the library builds with -fmad=false) plus the double-evaluated,
//     rounded sincos of the step kernel for headings and rays, so the numpy restatement gives the same bits.
//     A body smaller than a pixel may cover no pixel centre and then does not show.
//
// One block draws one tile (<= RND_PX pixels: whole rows, or one 1024-pixel piece of a row when W > 1024) of
// one environment.  It stages the environment's primitives in shared memory, top layer first, from the
// capacity slots of every list (one memory round trip, as k_lidar does), keeping only those whose bounding box
// reaches the tile; every pixel then takes the colour of the first primitive that covers it, which is what
// painting the layers bottom-up would leave.  The tile's bytes are assembled in shared memory at the output's
// alignment and stored with 16-byte stores (single bytes only at the ends of the tile's byte range).
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>
#include "msv_launch.h"

// The colour table, in the order masurv.h documents (msv_render_palette exports it).
#define MSV_PALETTE_INIT {                                                                   \
  {24, 26, 33},    /* background */            {196, 192, 178}, /* floor */                 \
  {224, 150, 130}, /* floor outside the zone */ {40, 150, 70},   /* zone ring */             \
  {235, 205, 50},  /* next-zone ring */        {92, 80, 70},    /* wall */                  \
  {235, 60, 160},  /* heal */                  {250, 150, 30},  /* box item */              \
  {140, 90, 45},   /* box */                                                                \
  {31, 119, 180}, {214, 39, 40}, {44, 160, 44}, {148, 103, 189},   /* agents 0-3 */          \
  {23, 190, 207}, {188, 189, 34}, {227, 119, 194}, {127, 127, 127}, /* agents 4-7 */         \
  {25, 70, 215},   /* team 0 */                {190, 20, 70},   /* team 1 */                \
  {255, 255, 255}, /* heading tick */          {0, 255, 140},   /* lidar ray */             \
}
enum { COL_BG = 0, COL_FLOOR, COL_OUTSIDE, COL_RING, COL_NEXT_RING, COL_WALL, COL_HEAL, COL_ITEM, COL_BOX,
       COL_AGENT0, COL_TEAM0 = COL_AGENT0 + 8, COL_TEAM1, COL_TICK, COL_RAY, N_COLOURS };
static const uint8_t h_palette[N_COLOURS][3] = MSV_PALETTE_INIT;
__constant__ uint8_t c_palette[N_COLOURS][3] = MSV_PALETTE_INIT;

#define RND_THREADS 256
#define RND_PX 1024                  // pixels per tile (4 per thread)
#define RND_MAXW 1024                // widest tile: a wider image is cut into row pieces of this width
// primitives of one environment: rays, ticks, agents, boxes, items, heals, walls, 2 rings, outside tint, floor
#define RND_SLOTS (MSV_MAX_AGENTS * MSV_MAX_LASERS + 2 * MSV_MAX_AGENTS + 2 * MSV_MAX_BOXES + MSV_MAX_HEALS + 8)
#define RND_CHUNKS ((RND_SLOTS + 31) / 32)
enum { P_CIRCLE = 0, P_RECT, P_RING, P_OUTSIDE, P_SEGMENT };

// sin and cos of a float angle evaluated in double and rounded to float -- the value b2Rot::Set gets in the step
// kernel (msv_device.cuh rot_sc) -- without the local-memory scratch array of the CUDA library's sincos (its
// Payne-Hanek path for large arguments).  The angle is reduced by pi/2 exactly in integer arithmetic: a float is
// m * 2^E with a 24-bit m, so 96 bits of 2/pi starting where m * 2^E * (2/pi) has weight 4 give the quadrant
// and a fraction good to 2^-70 for every finite float.  The fraction times pi/2 then goes through fdlibm's
// __kernel_sin / __kernel_cos polynomials (< 1 ulp on [-pi/4, pi/4]).  Rounded to float, the result equals the
// correctly rounded one except within ~2 double ulps of a float rounding boundary.
#define MSV_TWO_OVER_PI {0xA2F9836Eu, 0x4E441529u, 0xFC2757D1u, 0xF534DDC0u, 0xDB629599u, 0x3C439041u, 0xFE5163ABu, 0xDEBBC561u}
__constant__ uint32_t c_two_over_pi[8] = MSV_TWO_OVER_PI;
[[maybe_unused]] static const uint32_t h_two_over_pi[8] = MSV_TWO_OVER_PI;
__host__ __device__ __forceinline__ void rnd_sincos(float angle, float& s_out, float& c_out) {
#ifdef __CUDA_ARCH__
  const uint32_t* T = c_two_over_pi;
#else
  const uint32_t* T = h_two_over_pi;
#endif
  const float ax = fabsf(angle);
  if (!(ax <= 3.4028235e38f)) { s_out = c_out = angle - angle; return; }    // inf, nan: nan
  double r = (double)ax;
  int q = 0;
  if (ax > 0.78539816f) {
    uint32_t bits; memcpy(&bits, &ax, 4);
    const int E = (int)(bits >> 23) - 150;                                  // ax = m * 2^E (ax is normal here)
    const uint64_t m = (bits & 0x7fffffu) | 0x800000u;
    const int i0 = E - 1 > 1 ? E - 1 : 1;                                   // first bit of 2/pi that matters (1-based)
    const int sh = i0 + 95 - E;                                             // Z = m * W * 2^-sh, 94 <= sh <= 120
    const int j = (i0 - 1) >> 5, o = (i0 - 1) & 31;
    uint32_t w[3];
    for (int k = 0; k < 3; ++k) w[k] = (uint32_t)((((uint64_t)T[j + k] << 32) | T[j + k + 1]) >> (32 - o));
    const uint64_t t0 = m * w[2], t1 = m * w[1] + (t0 >> 32), hi = m * w[0] + (t1 >> 32);
    const uint64_t lo = (t1 << 32) | (t0 & 0xffffffffu);                    // P = hi * 2^64 + lo
    const int u = sh - 64;                                                  // 30..56
    q = (int)(hi >> u) & 3;
    const uint64_t fh = hi & ((1ull << u) - 1ull);
    double f = (double)fh * ldexp(1.0, -u) + (double)lo * ldexp(1.0, -sh);  // fraction of a quarter turn
    if (f >= 0.5) { f -= 1.0; q = (q + 1) & 3; }
    r = f * 1.57079632679489655800e+00 + f * 6.12323399573676603587e-17;   // f * pi/2
  }
  const double z = r * r;
  const double sn = r + (z * r) * (-1.66666666666666324348e-01 + z * (8.33333333332248946124e-03 + z * (-1.98412698298579493134e-04 +
                    z * (2.75573137070700676789e-06 + z * (-2.50507602534068634195e-08 + z * 1.58969099521155010221e-10)))));
  const double cr = z * (4.16666666666666019037e-02 + z * (-1.38888888888741095749e-03 + z * (2.48015872894767294178e-05 +
                    z * (-2.75573143513906633035e-07 + z * (2.08757232129817482790e-09 + z * -1.13596475577881948265e-11)))));
  const double hz = 0.5 * z, wc = 1.0 - hz;
  const double cs = wc + (((1.0 - wc) - hz) + z * cr);
  double s_ = q == 0 ? sn : q == 1 ? cs : q == 2 ? -sn : -cs;
  const double c_ = q == 0 ? cs : q == 1 ? -sn : q == 2 ? -cs : sn;
  if (signbit(angle)) s_ = -s_;
  s_out = (float)s_; c_out = (float)c_;
}

__device__ __forceinline__ float pix_x(int i, int W, float s) { return ((float)(2 * i - W + 1) * 0.5f) * s; }
__device__ __forceinline__ float pix_y(int j, int H, float s) { return ((float)(H - 1 - 2 * j) * 0.5f) * s; }

// Primitive records: a = (x0, y0, p, q), b = (len2, w2, kind, colour)
//   P_CIRCLE  (cx, cy, r*r)          dx*dx + dy*dy <= r*r
//   P_RECT    (cx, cy, hx, hy)       |x - cx| <= hx && |y - cy| <= hy
//   P_RING    (cx, cy, lo*lo, hi*hi) lo*lo <= d2 <= hi*hi
//   P_OUTSIDE (cx, cy, r*r, F/2)     on the floor and d2 > r*r
//   P_SEGMENT (px, py, ex, ey), b = (ex*ex + ey*ey, w*w): squared distance to the segment p .. p + e <= w*w
__device__ __forceinline__ bool covers(const float4 a, const float4 b, float x, float y) {
  const int kind = __float_as_int(b.z);
  const float dx = x - a.x, dy = y - a.y;
  if (kind == P_RECT) return fabsf(dx) <= a.z && fabsf(dy) <= a.w;
  if (kind == P_SEGMENT) {
    float t = 0.0f;
    if (b.x != 0.0f) t = fminf(fmaxf((dx * a.z + dy * a.w) / b.x, 0.0f), 1.0f);
    const float qx = dx - t * a.z, qy = dy - t * a.w;
    return qx * qx + qy * qy <= b.y;
  }
  const float d2 = dx * dx + dy * dy;
  if (kind == P_CIRCLE) return d2 <= a.z;
  if (kind == P_RING) return a.z <= d2 && d2 <= a.w;
  return fabsf(x) <= a.w && fabsf(y) <= a.w && d2 > a.z;   // P_OUTSIDE
}

__global__ void __launch_bounds__(RND_THREADS)
k_render(const __grid_constant__ DevConst C, const __grid_constant__ DevState S, const __grid_constant__ DevOut O,
         const __grid_constant__ RenderArgs R) {
  __shared__ float4 tab[RND_SLOTS][2];
  __shared__ __align__(16) uint8_t pix[3 * RND_PX + 16];
  __shared__ int chunk_n[RND_CHUNKS];
  __shared__ uint32_t pal[N_COLOURS];                // r | g << 8 | b << 16
  if (threadIdx.x < N_COLOURS)
    pal[threadIdx.x] = c_palette[threadIdx.x][0] | (uint32_t)c_palette[threadIdx.x][1] << 8 | (uint32_t)c_palette[threadIdx.x][2] << 16;
  const int A = C.A, N = C.N, L = R.lidar ? C.lidar_n : 0;
  const int nRay = A * L, oTick = nRay, oAgent = oTick + A, oBox = oAgent + A, oItem = oBox + R.BC, oHeal = oItem + R.BC;
  const int oWall = oHeal + R.HC, oNext = oWall + 4, T = oNext + 4;   // then: current ring, outside tint, floor
  const float s = R.s, hf = R.half_floor;
  for (int img = blockIdx.y; img < R.count; img += gridDim.y) {   // grid: x = tile of the image, y = images
    const int e = R.first + img, ti = blockIdx.x;
    const int ty = ti / R.tiles_x, tx = ti - ty * R.tiles_x;
    const int c0 = tx * R.TW, r0 = ty * R.TR;
    const int tw = min(R.TW, R.W - c0), th = min(R.TR, R.H - r0), npx = tw * th;
    // world rectangle of the tile's pixel centres
    const float xlo = pix_x(c0, R.W, s), xhi = pix_x(c0 + tw - 1, R.W, s);
    const float yhi = pix_y(r0, R.H, s), ylo = pix_y(r0 + th - 1, R.H, s);
    // ---- stage: one primitive per slot, top layer first; cull against the tile; compact in slot order
    for (int base = 0; base < T; base += RND_THREADS) {
      const int k = base + threadIdx.x;
      bool keep = false;
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = make_float4(0.f, 0.f, 0.f, 0.f);
      float bx0 = 0.f, bx1 = 0.f, by0 = 0.f, by1 = 0.f;   // bounding box
      int kind = P_CIRCLE, col = COL_BG;
      if (k < T) {
        const int counts = S.hdr0[e].x;
        if (k < oAgent) {                                // ray (agent i, ray r) or heading tick of agent i, reversed
          const bool ray = k < oTick;
          const int q = ray ? nRay - 1 - k : 0, i = ray ? q / L : A - 1 - (k - oTick), r = ray ? q - i * L : 0;
          const float4 k0 = S.akin0[i * N + e];
          keep = (__float_as_int(S.akin1[i * N + e].w) & 1) != 0;
          float ex, ey, w;
          if (ray) {                                     // k_lidar: off = from_polar(depth, (float)(ang + heading))
            const float frac = O.lidar_frac[((size_t)e * A + i) * R.LS + r];
            float sn, cs; rnd_sincos((float)(C.lidar_ang[r] + (double)k0.z), sn, cs);
            const float L0 = C.lidar_depth;
            const float offx = cs * L0 + (-sn) * 0.0f, offy = sn * L0 + cs * 0.0f;
            ex = (k0.x + frac * offx) - k0.x; ey = (k0.y + frac * offy) - k0.y;
            w = 0.5f * s; col = COL_RAY;
          } else {
            float sn, cs; rnd_sincos(k0.z, sn, cs);
            ex = (k0.x + C.agent_r * cs) - k0.x; ey = (k0.y + C.agent_r * sn) - k0.y;
            w = fmaxf(s, 0.2f * C.agent_r); col = COL_TICK;
          }
          kind = P_SEGMENT;
          a = make_float4(k0.x, k0.y, ex, ey); b = make_float4(ex * ex + ey * ey, w * w, 0.f, 0.f);
          bx0 = fminf(k0.x, k0.x + ex) - w; bx1 = fmaxf(k0.x, k0.x + ex) + w;
          by0 = fminf(k0.y, k0.y + ey) - w; by1 = fmaxf(k0.y, k0.y + ey) + w;
        } else if (k < oBox) {                           // agent
          const int i = A - 1 - (k - oAgent);
          const float4 k0 = S.akin0[i * N + e];
          keep = (__float_as_int(S.akin1[i * N + e].w) & 1) != 0;
          col = C.teams ? (i < A / 2 ? COL_TEAM0 : COL_TEAM1) : COL_AGENT0 + i;   // team rule of the observation
          const float rr = C.agent_r;
          a = make_float4(k0.x, k0.y, rr * rr, 0.f);
          bx0 = k0.x - rr; bx1 = k0.x + rr; by0 = k0.y - rr; by1 = k0.y + rr;
        } else if (k < oItem) {                          // box
          const int j = R.BC - 1 - (k - oBox);
          const float4 b0 = S.box0[j * N + e];
          keep = j < (counts & 255);
          kind = P_RECT; col = COL_BOX;
          a = b0;
          bx0 = b0.x - b0.z; bx1 = b0.x + b0.z; by0 = b0.y - b0.w; by1 = b0.y + b0.w;
        } else if (k < oWall) {                          // box item (its sensor circle) or heal
          const bool item = k < oHeal;
          const int j = item ? R.BC - 1 - (k - oItem) : R.HC - 1 - (k - oHeal);
          float2 c;
          if (item) { const float4 i0 = S.item0[j * N + e]; c = make_float2(i0.x, i0.y); }
          else c = S.heal[j * N + e];
          keep = j < (item ? (counts >> 8) & 255 : (counts >> 16) & 255);
          col = item ? COL_ITEM : COL_HEAL;
          const float rr = item ? C.item_r : C.heal_r;
          a = make_float4(c.x, c.y, rr * rr, 0.f);
          bx0 = c.x - rr; bx1 = c.x + rr; by0 = c.y - rr; by1 = c.y + rr;
        } else if (k < oNext) {                          // wall W, N, E, S (WallC order), reversed.  The walls' float
          const int j = 3 - (k - oWall);                 // rotation of (float)(pi/2) is ignored: W/E are drawn with
          const float hx = (j & 1) ? C.wall_hy : C.wall_hx, hy = (j & 1) ? C.wall_hx : C.wall_hy;   // half extents
          keep = true; kind = P_RECT; col = COL_WALL;    // (wall_hx, wall_hy), N/S with the two swapped
          a = make_float4(C.walls[j].px, C.walls[j].py, hx, hy);
          bx0 = a.x - hx; bx1 = a.x + hx; by0 = a.y - hy; by1 = a.y + hy;
        } else {                                         // next ring, current ring, outside tint, floor
          const int j = k - oNext;
          keep = true;
          if (j == 3) {
            kind = P_RECT; col = COL_FLOOR;
            a = make_float4(0.f, 0.f, hf, hf);
          } else if (j == 2) {
            const float4 zc = S.zonecur[e];
            kind = P_OUTSIDE; col = COL_OUTSIDE;
            a = make_float4(zc.x, zc.y, zc.z * zc.z, hf);
          } else {
            float cx, cy, rz;
            if (j == 1) { const float4 zc = S.zonecur[e]; cx = zc.x; cy = zc.y; rz = zc.z; col = COL_RING; }
            else {                                       // the `zone` observation's next zone: zonec[phase + 1]
              const int ph = S.zoneint[e].x;
              float2 zn = make_float2(0.f, 0.f);
              for (int z = 1; z < C.n_zones; ++z) { const float2 v = S.zonec[z * N + e]; if (z == ph + 1) zn = v; }
              keep = ph < C.zone_phases - 1;
              cx = zn.x; cy = zn.y; rz = keep ? C.zone_r32[ph + 1] : 0.f; col = COL_NEXT_RING;
            }
            const float lo = fmaxf(rz - s, 0.0f), hi = rz + s;
            kind = P_RING;
            a = make_float4(cx, cy, lo * lo, hi * hi);
            bx0 = cx - hi; bx1 = cx + hi; by0 = cy - hi; by1 = cy + hi;
          }
          if (j >= 2) { bx0 = -hf; bx1 = hf; by0 = -hf; by1 = hf; }
        }
        // conservative: a pixel centre the exact predicate accepts lies inside the box up to rounding
        const float sl = 1e-4f * (1.0f + fabsf(bx0) + fabsf(bx1) + fabsf(by0) + fabsf(by1));
        keep = keep && bx0 - sl <= xhi && bx1 + sl >= xlo && by0 - sl <= yhi && by1 + sl >= ylo;
      }
      const unsigned m = __ballot_sync(0xffffffffu, keep);
      if ((threadIdx.x & 31) == 0 && k < T) chunk_n[k >> 5] = __popc(m);
      __syncthreads();
      if (keep) {
        int off = __popc(m & ((1u << (threadIdx.x & 31)) - 1u));
        for (int c = 0; c < (k >> 5); ++c) off += chunk_n[c];
        b.z = __int_as_float(kind); b.w = __int_as_float(col);
        tab[off][0] = a; tab[off][1] = b;
      }
    }
    __syncthreads();
    int n = 0;
    for (int c = 0; c < (T + 31) >> 5; ++c) n += chunk_n[c];
    // ---- pixels: first covering primitive, top layer first
    uint8_t* const dst = R.out + (((size_t)img * R.H + r0) * R.W + c0) * 3;   // the tile's bytes are contiguous
    const int sh = (int)((uintptr_t)dst & 15);                               // staged at the output's alignment
    for (int p = threadIdx.x; p < npx; p += RND_THREADS) {
      const int row = p / tw, c = p - row * tw;
      const float x = pix_x(c0 + c, R.W, s), y = pix_y(r0 + row, R.H, s);
      int col = COL_BG;
      for (int q = 0; q < n; ++q) {
        const float4 a = tab[q][0], b = tab[q][1];
        if (covers(a, b, x, y)) { col = __float_as_int(b.w); break; }
      }
      const uint32_t v = pal[col];
      uint8_t* o = pix + sh + 3 * p;
      o[0] = (uint8_t)v; o[1] = (uint8_t)(v >> 8); o[2] = (uint8_t)(v >> 16);
    }
    __syncthreads();
    // ---- store: 16-byte words wholly inside the tile's byte range, single bytes at its two ends
    const int nb = 3 * npx, end = sh + nb;
    const int w0 = (sh + 15) >> 4, w1 = end >> 4;
    const int lo = min(w0 << 4, end), hi = max(w1 << 4, lo);
    uint8_t* const abase = dst - sh;
    for (int w = w0 + threadIdx.x; w < w1; w += RND_THREADS)
      reinterpret_cast<uint4*>(abase)[w] = reinterpret_cast<const uint4*>(pix)[w];
    const int nhead = lo - sh, ntail = end - hi;
    if ((int)threadIdx.x < nhead) abase[sh + threadIdx.x] = pix[sh + threadIdx.x];
    else if ((int)threadIdx.x >= 32 && (int)threadIdx.x < 32 + ntail) abase[hi + threadIdx.x - 32] = pix[hi + threadIdx.x - 32];
    __syncthreads();                                                         // (the next image reuses tab and pix)
  }
}

cudaError_t msv_launch_render(const DevConst& C, const DevState& S, const DevOut& O, RenderArgs R, cudaStream_t st) {
  R.TW = R.W < RND_MAXW ? R.W : RND_MAXW;
  R.TR = RND_PX / R.TW; if (R.TR > R.H) R.TR = R.H;
  R.tiles_x = (R.W + R.TW - 1) / R.TW;
  R.tiles_per_img = R.tiles_x * ((R.H + R.TR - 1) / R.TR);
  const float V = (float)(C.floor_size / 2 + C.floor_size / 100);
  R.s = (2.0f * V) / (float)(R.W < R.H ? R.W : R.H);
  R.half_floor = (float)(C.floor_size / 2);
  const dim3 grid((unsigned)R.tiles_per_img, (unsigned)(R.count < 65535 ? R.count : 65535));
  k_render<<<grid, RND_THREADS, 0, st>>>(C, S, O, R);
  return cudaPeekAtLastError();
}

int msv_palette(uint8_t* out_rgb, int capacity) {
  for (int k = 0; k < N_COLOURS && k < capacity; ++k)
    for (int c = 0; c < 3; ++c) out_rgb[3 * k + c] = h_palette[k][c];
  return N_COLOURS;
}
