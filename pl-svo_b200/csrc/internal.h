// internal.h — kernel argument blocks and launch entry points shared by the .cu files.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/plsvo_b200.h"

namespace plsvo {

constexpr int kCacheRows = 12;  // float4 rows per patch: 4 ref + 4 dx + 4 dy

// Device-layout description of one alignment batch (all pointers are device pointers).
struct AlignArgs {
  int B, n_pts, n_segs;
  int max_level, min_level, n_iter;
  double eps;
  int width, height;
  double fx, fy, cx, cy;
  // pyramid level l of pair b: img[l] + b*stride[l], rows pitch[l] bytes (pitch multiple of 16)
  const uint8_t* ref_img[PLSVO_MAX_LEVELS];
  const uint8_t* cur_img[PLSVO_MAX_LEVELS];
  uint32_t pitch[PLSVO_MAX_LEVELS];
  size_t stride[PLSVO_MAX_LEVELS];
  uint8_t img_in_smem[PLSVO_MAX_LEVELS];  // stage the cur level in shared memory with a bulk copy
  const double* T_ref_w;
  const double* T_cur_w;
  const int32_t* pt_count;
  const double* pt_px;
  const double* pt_f;
  const double* pt_pos;
  const uint8_t* pt_valid;
  const int32_t* seg_count;
  const double* seg_spx;
  const double* seg_epx;
  const double* seg_sf;
  const double* seg_ef;
  const double* seg_spos;
  const double* seg_epos;
  const double* seg_length;
  const uint8_t* seg_valid;
  const double* pt_depth;    // optional: |pos - ref_pos| per point (then pt_pos may be null)
  const double* seg_sdepth;  // optional: per segment start / end point
  const double* seg_edepth;
  // outputs
  double* out_T;
  long long* out_n_tracked;
  double* out_H;
  uint8_t* out_seg_killed;
  int32_t* out_iters;
  int32_t* out_status;
  uint32_t* out_patch_iters;
  uint32_t* out_patch_levels;
  // work distribution + per-CTA workspace
  unsigned int* work_counter;
  // arrival gate of the host-buffer pipeline: pair b may be touched once *arrived > b / gate_chunk
  // (a copy stream bumps it after each chunk of the batch has landed); gate_chunk == 0: no gate.
  const unsigned int* arrived;
  int gate_chunk;
  int max_patches;      // patch slots per pair: n_pts + max segment samples
  int max_seg_patches;  // segment sample slots per pair
  int max_seg_slots;    // lane slots of the segment groups per pair (multiple of 32)
  int smem_img_bytes;   // bytes of the image staging buffer
  float4* ws_cache;     // [grid][kCacheRows][max_patches] reference-patch cache (ref, dx, dy rows), L2 resident
  double* ws_segpx;     // [grid][2][max_seg_patches] 2-D centre of every segment sample (precompute only)
  double* ws_rec;       // [grid][5][rec_cap*threads] parked in-patch sums of segments longer than a warp
  int rec_cap;          // 32-sample trips of the longest segment, <= 32
  int derive_from;      // >= 0: the CTA forms levels (derive_from, max_level] of its pair by halfSample (gated pipeline)
  float one;            // 1.0f, deliberately a run-time value (device_math.cuh: add2_after_mul)
  // level units (DESIGN.md §4.1): the work queue hands out (pair, level) tickets, level-major, instead of whole pairs.
  // A pair's state between two levels goes through unit_state; unit_done[b] = (unit_epoch << 4) | levels of pair b done.
  int level_units;
  unsigned long long unit_epoch;  // counts the launches of the context from 1 (the words are cleared to 0 when allocated)
  unsigned long long* unit_done;  // [B]
  unsigned char* unit_state;     // [B][unit_state_stride]: AlignUnitState, pt_vis[n_pts], seg_alive[n_segs]
  size_t unit_state_stride;
};

// What a pair carries from one Gauss-Newton level to the next; everything else is rebuilt at the start of a level or
// recomputed from the inputs with identical bits.
struct AlignUnitState {
  double model[7], R[9], t[3];
  double chi2_prev;
  double H_last[36];
  long long n_meas_last;
  int stop, chi2_flags;
  unsigned int patch_iters, patch_levels;
  int iters_level[PLSVO_MAX_LEVELS];
};
inline size_t align_unit_state_stride(int n_pts, int n_segs) {
  return (sizeof(AlignUnitState) + (size_t)n_pts + (size_t)n_segs + 127) / 128 * 128;
}

// shared memory the kernel needs for a configuration (host + device agree through this)
size_t align_smem_bytes(int n_pts, int n_segs, int max_patches, int max_seg_slots, int img_bytes, int threads);
// kernel variants are compiled per (threads per CTA, resident CTAs per SM the register budget allows):
// (64,8) (96,7) (96,5) (128,5) (128,4) (160,3) (192,2) (256,2)
cudaError_t align_kernel_prepare(int threads, int min_blocks, size_t smem_bytes, int* ctas_per_sm);
cudaError_t weight_selftest_launch(uint32_t n, uint32_t seed, unsigned long long* d_mismatch, cudaStream_t s);
cudaError_t align_kernel_launch(const AlignArgs& a, int grid, int threads, int min_blocks, size_t smem_bytes,
                                cudaStream_t s);

// ---------------------------------------------------------------------------------------------
struct PoseOptArgs {
  int B, n_pts, n_segs;
  double fx, reproj_thresh;
  int n_iter, n_iter_ref;
  const double* T_f_w;
  const int32_t* pt_count;
  const double* pt_f;
  const double* pt_pos;
  const int32_t* pt_level;
  const uint8_t* pt_valid;
  const int32_t* seg_count;
  const double* seg_line;
  const double* seg_spos;
  const double* seg_epos;
  const int32_t* seg_level;
  const uint8_t* seg_valid;
  double* out_T;
  double* out_cov;
  double* out_scale;
  double* out_err_init;
  double* out_err_final;
  long long* out_num_pt;
  long long* out_num_ls;
  uint8_t* out_pt_outlier;
  uint8_t* out_seg_outlier;
  int32_t* out_iters;
  int32_t* out_status;
};
size_t poseopt_smem_bytes(int n_pts, int n_segs);
cudaError_t poseopt_kernel_launch(const PoseOptArgs& a, size_t smem_bytes, cudaStream_t s);


// ---------------------------------------------------------------------------------------------
struct PyramidArgs {
  int B, width, height, n_levels;  // n_levels <= 7 (64x64 level-0 tiles)
  uint8_t* level[PLSVO_MAX_LEVELS];  // device, [B][rows_l][pitch_l]; level[0] is the input
  uint32_t pitch[PLSVO_MAX_LEVELS];
  size_t stride[PLSVO_MAX_LEVELS];
};
cudaError_t pyramid_kernel_launch(const PyramidArgs& a, cudaStream_t s);


// ---------------------------------------------------------------------------------------------
struct Align2DArgs {
  int n, n_iter, width, height;
  const uint8_t* img[PLSVO_MAX_LEVELS];  // device, [n_images][rows_l][pitch_l]
  uint32_t pitch[PLSVO_MAX_LEVELS];
  size_t stride[PLSVO_MAX_LEVELS];
  const int32_t* image_index;
  const int32_t* level;
  const uint8_t* ref_patch_with_border;  // [n][100]
  const uint8_t* ref_patch;              // [n][64]
  const double* px;                      // [n][2]
  double* out_px;
  uint8_t* out_converged;
  const float* dir;   // align1D only: [n][2]
  double* out_h_inv;  // align1D only: [n]
};
cudaError_t align2d_kernel_launch(const Align2DArgs& a, cudaStream_t s);
cudaError_t align1d_kernel_launch(const Align2DArgs& a, cudaStream_t s);

// ---------------------------------------------------------------------------------------------
struct MatchArgs {
  int n, n_iter, n_pyr_levels, width, height;
  double fx, fy, cx, cy;
  const uint8_t* ref_img[PLSVO_MAX_LEVELS];  // device, [n_ref][rows_l][pitch_l]
  uint32_t ref_pitch[PLSVO_MAX_LEVELS];
  size_t ref_stride[PLSVO_MAX_LEVELS];
  const uint8_t* cur_img[PLSVO_MAX_LEVELS];
  uint32_t cur_pitch[PLSVO_MAX_LEVELS];
  size_t cur_stride[PLSVO_MAX_LEVELS];
  const double* T_ref_w;  // [n_ref][7]
  const double* T_cur_w;  // [n_cur][7]
  const int32_t* ref_index;
  const int32_t* cur_index;
  const double* ref_px;
  const double* ref_f;
  const int32_t* ref_level;
  const uint8_t* is_edgelet;  // may be null
  const double* ref_grad;     // may be null
  const double* pos;
  const double* px_cur;
  double* out_px;
  uint8_t* out_success;
  int32_t* out_level;
  double* out_A;  // [n][4] or null
};
cudaError_t match_direct_kernel_launch(const MatchArgs& a, cudaStream_t s);

// ---------------------------------------------------------------------------------------------
struct SeedArgs {
  int n, n_iter, n_pyr_levels, width, height, max_epi_search_steps;
  int spw;           // seeds per warp (set by the launch functions)
  int serial_steps;  // steps of an epipolar search walked by the seed's own thread before the warp takes over
  int align_1d, subpix_refinement, edgelet_filtering;
  double edgelet_max_angle, convergence_thresh;
  double fx, fy, cx, cy;
  const uint8_t* ref_img[PLSVO_MAX_LEVELS];
  uint32_t ref_pitch[PLSVO_MAX_LEVELS];
  size_t ref_stride[PLSVO_MAX_LEVELS];
  const uint8_t* cur_img[PLSVO_MAX_LEVELS];
  uint32_t cur_pitch[PLSVO_MAX_LEVELS];
  size_t cur_stride[PLSVO_MAX_LEVELS];
  const double* T_ref_w;
  const double* T_cur_w;
  const int32_t* ref_index;
  const int32_t* cur_index;
  const double* ref_px;
  const double* ref_f;
  const int32_t* ref_level;
  const uint8_t* is_edgelet;  // may be null
  const double* ref_grad;     // may be null
  const float* a;
  const float* b;
  const float* mu;
  const float* z_range;
  const float* sigma2;
  // line seeds only
  const double* ref_sf;
  const double* ref_ef;
  const float* mu_e;
  const float* z_range_e;
  const float* sigma2_e;
  float* out_mu_e;
  float* out_sigma2_e;
  double* out_depth_e;
  double* out_px_cur_e;  // [n][2]
  float* out_a;
  float* out_b;
  float* out_mu;
  float* out_sigma2;
  int32_t* out_status;
  uint8_t* out_converged;
  double* out_depth;
  double* out_px_cur;
};
cudaError_t seed_update_kernel_launch(const SeedArgs& a, cudaStream_t s);
cudaError_t line_seed_update_kernel_launch(const SeedArgs& a, cudaStream_t s);

// ---------------------------------------------------------------------------------------------
struct StructOptArgs {
  int n_points, n_segs, n_iter_pts, n_iter_segs;
  const double* T_f_w;
  const int32_t* pt_obs_begin;
  const int32_t* pt_obs_frame;
  const double* pt_obs_f;
  const double* pt_pos;
  const int32_t* seg_obs_begin;
  const int32_t* seg_obs_frame;
  const double* seg_obs_sf;
  const double* seg_obs_ef;
  const double* seg_spos;
  const double* seg_epos;
  double* out_pt_pos;
  double* out_seg_spos;
  double* out_seg_epos;
  int32_t* out_pt_iters;
  int32_t* out_seg_iters;
};
cudaError_t structopt_kernel_launch(const StructOptArgs& a, cudaStream_t s);

}  // namespace plsvo
