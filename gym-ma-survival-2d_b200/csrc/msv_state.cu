// msv_state.cu -- the global state of every environment (msv_enable_global_state): one float32 row of Ds floats
// per environment, what an omniscient observer sees stored once (the agents' rows and alive mask, the zone,
// the heals, boxes and floor box items with their presence masks, every agent's inventory top), then the step
// count.  The layout is gs_layout() (msv_launch.h); include/masurv.h and DESIGN.md §2 document it.
//
// k_global_state is k_obs2's source-major scheme for one output: a block is a tile of 32 consecutive environments
// (lane = environment: the SoA loads are fully coalesced), a warp takes one source item -- agent j, box k, floor
// item k, heal k, or the zone and step count -- and scatters its values into a shared-memory stage [32][Dsp]
// (Dsp = Ds rounded up to an odd number: the 32 lanes' stores of one column hit 32 different banks).  The tile's
// rows are ONE contiguous run of rows * Ds floats at e0 * Ds, 16-byte aligned (e0 and rows are multiples of 4),
// copied out with 16-byte stores.
// kRows (terminal capture): only the rows of real environments whose only_if byte is set are written, with scalar
// stores; every other row is left untouched, and a tile without such a row leaves at once.
#include <cuda_runtime.h>
#include <stdint.h>
#include "msv_launch.h"

#define GS_E 32                 // environments per tile
#define GS_MAX_DS (MSV_MAX_AGENTS * 10 + 6 + 3 * MSV_MAX_HEALS + 2 * MSV_MAX_AGENTS + 23 * MSV_MAX_BOXES + 9 * MSV_MAX_AGENTS + 1)

template <bool kRows>
__global__ void __launch_bounds__(1024)
k_global_state(const __grid_constant__ DevConst C, const __grid_constant__ DevState S, const __grid_constant__ GsLayout Lg,
               float* __restrict__ out, const uint8_t* __restrict__ only_if) {
  extern __shared__ float stage[];
  // the next step's k_step may be launched programmatically dependent on this kernel: let it become resident (its
  // griddepcontrol.wait still waits for this grid to complete before it touches the state)
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const int A = C.A, B = C.B0, H = C.H0, Sw = C.S, N = C.N, Ds = Lg.Ds, Dsp = Ds | 1;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int e0 = blockIdx.x * GS_E, e = e0 + lane;
  const int rows = N - e0 < GS_E ? N - e0 : GS_E;    // N is a multiple of the step kernel's tile, itself a multiple of 4
  const bool live = lane < rows;
  unsigned sel = 0u;                                  // kRows: bit r = row r is written (every warp computes the same mask)
  if (kRows) {
    sel = __ballot_sync(0xffffffffu, live && e < C.n_real && only_if[e] != 0);
    if (!sel) return;
  }
  float* const row = stage + lane * Dsp;
  // b2PolygonShape vertex order (Q8): a copy of k_obs2's vert (msv_kernels.cu), so that k_obs2 stays as it is
  auto vert = [&](float hx, float hy, int rot, int comp) {
    int j = ((comp >> 1) + rot) & 3;
    return (comp & 1) ? ((j >= 2) ? hy : -hy) : ((j == 1 || j == 2) ? hx : -hx);
  };
  const int n_items = A + 2 * B + H + 1, nwarps = blockDim.x >> 5;
  // (state loads bypass L1 -- __ldcg: each word is read once)
  for (int it = warp; it < n_items; it += nwarps) {
    if (!live) continue;
    if (it < A) {                                     // ---- agent j: its row, alive flag and inventory top
      const int j = it;
      const float4 k0 = __ldcg(&S.akin0[j * N + e]), k1 = __ldcg(&S.akin1[j * N + e]); const int4 ai = __ldcg(&S.aint[j * N + e]);
      const bool al = (__float_as_int(k1.w) & 1) != 0;
      const int inv = ai.w, n = inv & 7, top = n > 0 ? (inv >> (4 + 2 * (n - 1))) & 3 : 0;
      const int tm = C.teams ? 1 : 0;
      float* r = row + Lg.col[GS_AGENTS] + j * Sw;    // [id, (team), health, x, y, angle, vx, vy, omega]; dead: id, team
      r[0] = (float)j; if (tm) r[1] = (float)(j < A / 2 ? 0 : 1);
      r[tm + 1] = al ? (float)ai.x : 0.f; r[tm + 2] = al ? k0.x : 0.f; r[tm + 3] = al ? k0.y : 0.f; r[tm + 4] = al ? k0.z : 0.f;
      r[tm + 5] = al ? k0.w : 0.f; r[tm + 6] = al ? k1.x : 0.f; r[tm + 7] = al ? k1.y : 0.f;
      row[Lg.col[GS_AGENTS_MASK] + j] = al ? 0.f : 1.f;
      if (H > 0) {
        const bool has = al && top == MSV_ITEM_HEAL;
        row[Lg.col[GS_HEAL_SLOT] + j] = has ? (float)C.healing : 0.f; row[Lg.col[GS_HEAL_SLOT_MASK] + j] = has ? 0.f : 1.f;
      }
      if (B > 0) {
        const bool has = al && top == MSV_ITEM_BOX;
        float4 pl = make_float4(0.f, 0.f, 0.f, 0.f);
        if (has) pl = __ldcg(&S.ainv[(j * 4 + n - 1) * N + e]);
        for (int c = 0; c < 8; ++c) row[Lg.col[GS_BOX_SLOT] + j * 8 + c] = has ? vert(pl.x, pl.y, __float_as_int(pl.w) & 1, c) : 0.f;
        row[Lg.col[GS_BOX_SLOT_MASK] + j] = has ? 0.f : 1.f;
      }
    } else if (it < A + B) {                          // ---- box k: vertices, x, y, angle (always 0)
      const int k = it - A;
      float4 b0 = make_float4(0.f, 0.f, 0.f, 0.f); int rot = 0;
      const bool on = k < (__ldcg(&S.hdr0[e].x) & 255);
      if (on) { b0 = __ldcg(&S.box0[k * N + e]); rot = (__ldcg(&S.box1[k * N + e].y) >> 1) & 1; }
      float* r = row + Lg.col[GS_BOXES] + k * 11;
      for (int c = 0; c < 8; ++c) r[c] = on ? vert(b0.z, b0.w, rot, c) : 0.f;
      r[8] = b0.x; r[9] = b0.y; r[10] = 0.f;
      row[Lg.col[GS_BOXES_MASK] + k] = on ? 0.f : 1.f;
    } else if (it < A + 2 * B) {                      // ---- floor box item k (always rotated)
      const int k = it - A - B;
      float4 i0 = make_float4(0.f, 0.f, 0.f, 0.f);
      const bool on = k < ((__ldcg(&S.hdr0[e].x) >> 8) & 255);
      if (on) i0 = __ldcg(&S.item0[k * N + e]);
      float* r = row + Lg.col[GS_BOX_ITEMS] + k * 10;
      for (int c = 0; c < 8; ++c) r[c] = on ? vert(i0.z, i0.w, 1, c) : 0.f;
      r[8] = i0.x; r[9] = i0.y;
      row[Lg.col[GS_BOX_ITEMS_MASK] + k] = on ? 0.f : 1.f;
    } else if (it < A + 2 * B + H) {                  // ---- heal k
      const int k = it - A - 2 * B;
      float2 hh = make_float2(0.f, 0.f);
      const bool on = k < ((__ldcg(&S.hdr0[e].x) >> 16) & 255);
      if (on) hh = __ldcg(&S.heal[k * N + e]);
      row[Lg.col[GS_HEALS] + 2 * k] = hh.x; row[Lg.col[GS_HEALS] + 2 * k + 1] = hh.y;
      row[Lg.col[GS_HEALS_MASK] + k] = on ? 0.f : 1.f;
    } else {                                          // ---- zone (current x, y, r; next x, y, r) and step count
      const float4 zc = __ldcg(&S.zonecur[e]); const int ph = __ldcg(&S.zoneint[e].x);
      float z3 = 0.f, z4 = 0.f, z5 = 0.f;
      if (ph < C.zone_phases - 1) { const float2 c2 = __ldcg(&S.zonec[(ph + 1) * N + e]); z3 = c2.x; z4 = c2.y; z5 = C.zone_r32[ph + 1]; }
      float* r = row + Lg.col[GS_ZONE];
      r[0] = zc.x; r[1] = zc.y; r[2] = zc.z; r[3] = z3; r[4] = z4; r[5] = z5;
      row[Lg.col[GS_STEPS]] = (float)__ldcg(&S.hdr0[e].y);
    }
  }
  __syncthreads();
  float* const dst = out + (size_t)e0 * Ds;
  if (kRows) {
    for (int q = threadIdx.x; q < rows * Ds; q += blockDim.x) {
      const int r = q / Ds;
      if ((sel >> r) & 1u) dst[q] = stage[r * Dsp + (q - r * Ds)];
    }
  } else {
    float4* const dst4 = reinterpret_cast<float4*>(dst);
    for (int q4 = threadIdx.x; q4 < rows * Ds / 4; q4 += blockDim.x) {
      int r = (4 * q4) / Ds, c = 4 * q4 - r * Ds;
      float v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        v[u] = stage[r * Dsp + c];
        if (++c == Ds) { c = 0; ++r; }
      }
      dst4[q4] = make_float4(v[0], v[1], v[2], v[3]);
    }
  }
}

static size_t gs_smem(int Ds) { return (size_t)GS_E * (Ds | 1) * sizeof(float); }

cudaError_t msv_global_state_attrs() {
  const int smem = (int)gs_smem(GS_MAX_DS);
  cudaError_t e = cudaFuncSetAttribute(k_global_state<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_global_state<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  return e;
}

cudaError_t msv_launch_global_state(const DevConst& C, const DevState& S, const GsLayout& Lg, float* out, const uint8_t* only_if,
                                    cudaStream_t st) {
  // one warp per source item when they fit a block (a single round of loads), else 32 warps looping over the items
  const int n_items = C.A + 2 * C.B0 + C.H0 + 1;
  const int threads = n_items <= 32 ? 32 * n_items : 1024;
  const unsigned grid = (unsigned)((C.N + GS_E - 1) / GS_E);
  if (only_if) k_global_state<true><<<grid, threads, gs_smem(Lg.Ds), st>>>(C, S, Lg, out, only_if);
  else k_global_state<false><<<grid, threads, gs_smem(Lg.Ds), st>>>(C, S, Lg, out, only_if);
  return cudaPeekAtLastError();
}
