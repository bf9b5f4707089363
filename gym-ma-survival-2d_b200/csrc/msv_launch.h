// msv_launch.h -- host-side interface between the C ABI (msv_abi.cu) and the
// kernel launchers (msv_kernels.cu, msv_render.cu, msv_state.cu).
#pragma once
#include "msv_types.cuh"
#define MSV_TPB 512   // maximum threads per block of k_step / k_reset / k_observe (the actual size is a runtime choice, see plan_blocks)
// cap: capacity class 0 = <2,4,4>, 1 = <4,4,4>, 2 = <8,8,16>; which: 0 step, 2 observe, 3 one-time kernel attribute setup
cudaError_t msv_launch(int cap, int which, const DevConst& C, const DevState& S, const DevOut& O,
                       const uint8_t* actions, cudaStream_t st);
// k_reset of the envs whose mask byte is set (mask NULL: every env).  finished != 0: the reset ends a finished
// episode (counted, outputs kept; the mask covers the padded batch); 0: a restart (not counted, the env's rewards,
// dones, truncated -- when not NULL -- and BattleRoyale flags are zeroed; the mask covers the real envs).
cudaError_t msv_launch_reset(int cap, const DevConst& C, const DevState& S, const DevOut& O, const uint8_t* mask, int finished,
                             uint8_t* truncated, cudaStream_t st);
// k_truncate: step limit T > 0 after a step without the in-kernel reset; writes truncated and finished (uint8[N])
cudaError_t msv_launch_truncate(const DevConst& C, const DevState& S, const DevOut& O, int T, uint8_t* truncated, uint8_t* finished,
                                cudaStream_t st);
void msv_capacity(int cap, int* AC, int* BC, int* HC, int* P, int* PW, int* sm_words);
cudaError_t msv_launch_stats(int N, int stride, int AC, float* sreward, int* skills, int4* smisc, double* out_reward,
                             unsigned long long* out_kills, unsigned long long* out_misc, cudaStream_t st);
cudaError_t msv_read_profile(unsigned long long out[64], int reset);
cudaError_t msv_read_blocks(unsigned long long* out, int n_words);
cudaError_t msv_read_trace(unsigned long long* out, int n_words);
cudaError_t msv_read_check(unsigned long long out[2]);
cudaError_t msv_launch_spare(const DevConst& C, const DevState& S, const uint8_t* dones, int only_done, cudaStream_t st);
// k_obs2 into T's tensors (F NULL) or into F's flat rows: every row (only_if NULL), or the rows of the real envs
// whose only_if byte is set
cudaError_t msv_launch_obs(const DevConst& C, const DevState& S, const ObsTable& T, const ObsFlat* F, int AC, const uint8_t* only_if,
                           cudaStream_t st);
// k_lidar; LS: floats between two agents' rows of O.lidar_frac (L in the dict layout, D in the flat one)
cudaError_t msv_launch_lidar(const DevConst& C, const DevState& S, const DevOut& O, int BC, int HC, int LS, cudaStream_t st);
// msv_render: picture of envs [first, first+count) into out (uint8[count][H][W][3]); BC, HC the list capacities,
// lidar != 0 draws the rays (LS: the row stride of O.lidar_frac, as k_lidar).  The launcher fills in the tiling
// and the viewport (the fields after `LS`).
struct RenderArgs {
  int first, count, H, W, BC, HC, lidar, LS;
  int TW, TR, tiles_x, tiles_per_img;   // tile width and rows, tiles per image row and per image
  float s, half_floor;                  // pixel size, floor_size / 2
  uint8_t* out;
};
cudaError_t msv_launch_render(const DevConst& C, const DevState& S, const DevOut& O, RenderArgs R, cudaStream_t st);
int msv_palette(uint8_t* out_rgb, int capacity);   // copies min(capacity, n) colours, returns n

// ---- global state (msv_state.cu) -------------------------------------------
// The row of one environment, keys in this order (a key whose list the config lacks has width 0: no heal keys when
// H = 0, no box keys when B = 0).  col[k] is key k's first column, Ds the row width.
enum { GS_AGENTS, GS_AGENTS_MASK, GS_ZONE, GS_HEALS, GS_HEALS_MASK, GS_HEAL_SLOT, GS_HEAL_SLOT_MASK, GS_BOXES,
       GS_BOXES_MASK, GS_BOX_ITEMS, GS_BOX_ITEMS_MASK, GS_BOX_SLOT, GS_BOX_SLOT_MASK, GS_STEPS, GS_KEYS };
struct GsLayout { int col[GS_KEYS]; int Ds; };
inline GsLayout gs_layout(int A, int B, int H, int S) {
  const int hk = H > 0 ? 1 : 0, bk = B > 0 ? 1 : 0;
  const int w[GS_KEYS] = {A * S, A, 6, hk * 2 * H, hk * H, hk * A, hk * A, bk * 11 * B, bk * B, bk * 10 * B, bk * B, bk * 8 * A, bk * A, 1};
  GsLayout L;
  int c = 0;
  for (int k = 0; k < GS_KEYS; ++k) { L.col[k] = c; c += w[k]; }
  L.Ds = c;
  return L;
}
// one-time, on the current device: the dynamic shared memory k_global_state's stage needs (up to 52 KB)
cudaError_t msv_global_state_attrs();
// k_global_state into out ([C.N][Ds] floats): every row (only_if NULL), or the rows of the real envs whose
// only_if byte is set
cudaError_t msv_launch_global_state(const DevConst& C, const DevState& S, const GsLayout& Lg, float* out, const uint8_t* only_if,
                                    cudaStream_t st);
