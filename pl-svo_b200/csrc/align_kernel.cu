// align_kernel.cu — sparse image alignment (plsvo::SparseImgAlign::run, src/sparse_img_align.cpp:54-95)
// as ONE persistent sm_100a kernel: a CTA owns a frame pair for its whole coarse-to-fine
// Gauss-Newton optimisation, so a pair costs no host round trips and no re-launches.
//
// Mapping (DESIGN.md §4.1):
//   * work queue: CTAs pull pair indices from an atomic counter (iteration counts vary per pair).
//   * per level: one thread issues a bulk async copy (TMA engine, cp.async.bulk -> UBLKCP) of the
//     current image level into shared memory while all threads precompute the reference-patch
//     cache (4x4 bilinear intensities + central-difference gradients: sparse_img_align.cpp:195-378)
//     from the reference image in global memory into a per-CTA, L2-resident workspace.
//   * per GN pass, phase 1 (residuals): thread per patch.  The patch centre is warped in double, the
//     4x4 residuals, robust weights and chi2 terms are evaluated in float with the reference's exact
//     operation order (:450-500 points, :612-637 segment samples), and the five in-patch sums
//     (w*dx*dx, w*dx*dy, w*dy*dy, w*dx*r, w*dy*r) are accumulated per pixel in DOUBLE, as the
//     reference accumulates every pixel's J*J^T*w in double (:487-492).
//   * chi2 is reproduced BIT-EXACTLY in the reference's order (float accumulator, points in list
//     order, pixels row-major, :484; then one term per segment, :683; pt_chi2 + seg_chi2, :171),
//     because the accept/rollback decision of vk::NLLSSolver (`new_chi2 > chi2_`) compares two such
//     sums that often agree to ~1e-6.  A sequential float sum is evaluated in parallel as follows:
//     while the running sum s stays inside one binade, s -> fl(s + t) only depends on the parity of
//     s's mantissa, so a patch's 16 additions collapse to "add A[parity] ulps"; these maps compose
//     associatively (segmented warp scan).  Each patch classifies itself from the exact prefix sum of
//     the patch totals (one block barrier per round of NT patches) with a rigorous error margin:
//     patches that may cross a power of two keep their 16 terms ("opaque", ~10 per pass) and are
//     chained serially by one warp together with the composed maps.
//   * phase 2 (normal equations): J_px = (dx*row0 + dy*row1)*fx/2^l (:261-262) factorises, so
//     H += [r0 r1] S [r0 r1]^T per patch — a rank-2 update of the thread's 21+6 double accumulators,
//     replacing the reference's 6x(N*16) double Jacobian cache (768 B/patch) by 128 B/patch of float
//     gradients.  Reduced with a register-halving warp shuffle tree, then across warps through shared
//     memory in fixed order (bitwise reproducible run to run).
//   * thread 0 solves the 6x6 system (LDLT), applies T <- T*exp(-x) and the vikit NLLSSolver
//     accept / rollback / convergence logic on chip while a second warp chains the chi2 items.
#include <cuda_runtime.h>
#include <stdint.h>

#include "device_math.cuh"
#include "internal.h"

namespace plsvo {

namespace {

constexpr int kOpqCap = 48;  // opaque patches (16 float terms each) per pass; one per binade crossing + margin

struct PairCtl {
  double R[9];
  double t[3];
  double model[7];      // T_cur_from_ref (q, t)
  double old_model[7];
  double T_ref[7];
  double ref_pos[3];
  double chi2_prev;
  double H_last[36];
  double scratch[36];
  double g[6];
  double x[6];
  unsigned long long mbar;
  long long n_meas_last;
  int pair;      // work-queue ticket of the current unit
  int level_lo;  // finest level of the current unit
  int flag;
  int stop;
  int iter;
  int n_seg_patches;
  int n_seg_slots;  // lane slots taken by the segment groups at the current level
  unsigned int patch_iters;
  unsigned int patch_levels;
  int iters_level[PLSVO_MAX_LEVELS];
  double cand[7];  // candidate model T*exp(-x) of the current pass and its rotation matrix / step norm
  double candR[9];
  double cand_nm;
  float seg_chi2f; // seg_chi2 of the current pass (:683), summed by a third warp while the walker chains the points
  float chi2f;     // chi2 of the current pass, summed in the reference's order (walker warp -> thread 0)
  int n_opq;       // opaque patches of the current pass
  int chi2_flags;  // sticky per pair: 1 = opaque buffer overflowed (order approximated), 2 = binade check failed
};

struct Layout {
  uint32_t ctl, red, tot, chunk_tot, items, cnt, flat, opq, seg_N0, seg_N, seg_off, seg_slot, slot_seg, seg_term,
      seg_alive, pt_vis, xyz, tsc, img, total;
};

__host__ __device__ inline uint32_t align_up(uint32_t v, uint32_t a) { return (v + a - 1) / a * a; }

__host__ __device__ inline Layout make_layout(int n_pts, int n_segs, int max_patches, int max_seg_slots, int img_bytes,
                                              int nt) {
  Layout L;
  const uint32_t nw = (uint32_t)nt / 32u;
  const uint32_t rounds = ((uint32_t)n_pts + (uint32_t)nt - 1u) / (uint32_t)nt;
  const uint32_t n_chunks = ((uint32_t)n_pts + 31u) / 32u;
  uint32_t o = 0;
  L.ctl = o;
  o = align_up(o + (uint32_t)sizeof(PairCtl), 16);
  L.red = o;
  o += nw * 32u * 8u;  // cross-warp partials
  L.tot = o;
  o += 32u * 8u;
  L.chunk_tot = o;
  o += 8u * (rounds * nw + 1u);  // per 32-patch chunk: float-chi2 total (estimate) of the pass
  L.items = o;
  o += 8u * 32u * (n_chunks + 1u);  // composed chi2 maps / opaque references, <= 32 per chunk
  L.cnt = o;
  o += 4u * (n_chunks + 1u);
  L.flat = align_up(o, 8);
  o = L.flat + 8u * 64u;  // the walker's current batch of items, in list order
  L.opq = align_up(o, 16);
  o = L.opq + 64u * (uint32_t)kOpqCap;
  L.seg_N0 = o;
  o += 4u * (uint32_t)n_segs;  // samples of every segment at level 0 (setupSampling), once per pair
  L.seg_N = o;
  o += 4u * (uint32_t)n_segs;
  L.seg_off = o;
  o += 4u * (uint32_t)n_segs;
  L.seg_slot = o;
  o += 4u * (uint32_t)n_segs;
  L.slot_seg = o;
  o += 2u * (uint32_t)max_seg_slots;  // lane slot -> segment (groups of 2^k lanes, k per segment)
  L.seg_term = align_up(o, 4);
  o = L.seg_term;
  o += 4u * (uint32_t)n_segs;  // per-segment chi2 term of the current pass (-1: none)
  L.seg_alive = o;
  o += (uint32_t)n_segs;
  L.pt_vis = o;
  o += (uint32_t)n_pts;
  L.xyz = align_up(o, 16);
  o = L.xyz + 3u * 8u * (uint32_t)max_patches;  // X/Z, Y/Z, 1/Z of every patch's 3-D point in the ref frame
  L.tsc = o;
  o += 16u * 4u * (uint32_t)nt;  // the 16 chi2 terms of each thread's current patch ([k][tid]: conflict-free)
  o = align_up(o, 128);
  L.img = o;
  o += (uint32_t)img_bytes + 16u;  // slack: the 5-byte row reads fetch whole aligned words
  L.total = o;
  return L;
}

// bilinear sample with the reference's operation order: ((wTL*a + wTR*b) + wBL*c) + wBR*d,
// every product and sum rounded separately (no FMA contraction) — sparse_img_align.cpp:458
__device__ __forceinline__ float bilin(float wTL, float wTR, float wBL, float wBR, float a, float b, float c, float d) {
  return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(wTL, a), __fmul_rn(wTR, b)), __fmul_rn(wBL, c)), __fmul_rn(wBR, d));
}

// Patch::setPosition + isInFrame + computeInterpWeights (src/feature.cpp:189-208, feature.h:139-144).
// The weights are computed in float: for accepted patches (floor >= boundary >= 2) 1-subpix is
// exact in float and each product is rounded once, which equals the reference's double-then-narrow.
__device__ __forceinline__ bool patch_setup(double u, double v, int cols, int rows, int boundary, int& ui, int& vi,
                                            float& wTL, float& wTR, float& wBL, float& wBR) {
  const float uf = (float)u, vf = (float)v;
  const float fu = floorf(uf), fv = floorf(vf);
  ui = (int)fu;
  vi = (int)fv;
  if (ui < boundary || vi < boundary || ui >= cols - boundary || vi >= rows - boundary) return false;
  const float su = __fsub_rn(uf, fu), sv = __fsub_rn(vf, fv);
  const float omu = __fsub_rn(1.0f, su), omv = __fsub_rn(1.0f, sv);
  wTL = __fmul_rn(omu, omv);
  wTR = __fmul_rn(su, omv);
  wBL = __fmul_rn(omu, sv);
  wBR = __fmul_rn(su, sv);
  return true;
}

// LineFeat::setupSampling (src/feature.cpp:160-173) followed by the per-level decimation (:320).
// The sample count is clamped to 2^20 like the host-side sizing (plsvo_abi.cu:host_seg_samples), so a
// non-finite or absurd length cannot overflow the int conversion.
__device__ __noinline__ int seg_num_samples0(const double* spx, const double* epx, double length) {
  const double a0 = fabs(epx[0] - spx[0]), a1 = fabs(epx[1] - spx[1]);
  // explicit round-to-nearest operations: the sample count is structural and must equal the reference's
  // (and the host-side sizing's) value, so nothing here may be contracted into an FMA
  const double tan_dir = __ddiv_rn(fmin(a0, a1), fmax(a0, a1));
  const double sin_dir = __ddiv_rn(tan_dir, __dsqrt_rn(__dadd_rn(1.0, __dmul_rn(tan_dir, tan_dir))));
  const double correction = __dmul_rn(2.0, __dsqrt_rn(__dadd_rn(1.0, __dmul_rn(sin_dir, sin_dir))));
  double nd = __ddiv_rn(length, __dmul_rn(8.0, correction));
  if (!(nd >= 1.0)) nd = 1.0;  // fmax(1, x) of the reference; also catches NaN
  if (nd > 1048576.0) nd = 1048576.0;
  return (int)(unsigned long long)nd;  // N_samples at level 0; level l uses 1 + (N0 - 1) / 2^l (:320)
}

__device__ __forceinline__ bool cam_in_frame(int ox, int oy, int boundary, int level, int width, int height) {
  return ox >= boundary && ox < width / (1 << level) - boundary && oy >= boundary &&
         oy < height / (1 << level) - boundary;
}

// vk::PinholeCamera::cam2world without distortion (rpg_vikit pinhole_camera.cpp; the constructors of PointFeat / LineFeat
// derive their bearing vectors this way, src/feature.cpp:42,98-99): ((u-cx)/fx, (v-cy)/fy, 1).normalized(), every
// operation rounded on its own (Eigen: x / sqrt(x.x)).
__device__ __forceinline__ void cam2world(const AlignArgs& a, const double* px, double* f) {
  const double x = __ddiv_rn(__dsub_rn(px[0], a.cx), a.fx), y = __ddiv_rn(__dsub_rn(px[1], a.cy), a.fy);
  const double n = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)), 1.0));
  f[0] = __ddiv_rn(x, n), f[1] = __ddiv_rn(y, n), f[2] = __ddiv_rn(1.0, n);
}

// Rank-2 update of the 21 (upper-triangular H) + 6 (Jres) accumulators of one thread for a patch whose 3-D
// point has normalised coordinates (xn, yn) = (X/Z, Y/Z) and inverse depth zi = 1/Z:
//   H += Sxx r0 r0^T + Sxy (r0 r1^T + r1 r0^T) + Syy r1 r1^T ,  Jres -= Sxr r0 + Syr r1
// with the rows of Frame::jacobian_xyz2uv (include/plsvo/frame.h:138-160) written in (xn, yn, zi).
__device__ __forceinline__ void rank2_update(double* acc, double xn, double yn, double zi, double Sxx, double Sxy,
                                             double Syy, double Sxr, double Syr) {
  double r0[6], r1[6];
  const double xy = xn * yn;
  r0[0] = -zi, r0[1] = 0.0, r0[2] = xn * zi, r0[3] = xy, r0[4] = -(1.0 + xn * xn), r0[5] = yn;
  r1[0] = 0.0, r1[1] = -zi, r1[2] = yn * zi, r1[3] = 1.0 + yn * yn, r1[4] = -xy, r1[5] = -xn;
  double p[6], q[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    p[i] = Sxx * r0[i] + Sxy * r1[i];
    q[i] = Sxy * r0[i] + Syy * r1[i];
  }
  int idx = 0;
#pragma unroll
  for (int i = 0; i < 6; ++i)
#pragma unroll
    for (int j = i; j < 6; ++j) acc[idx++] += p[i] * r0[j] + q[i] * r1[j];
#pragma unroll
  for (int i = 0; i < 6; ++i) acc[21 + i] -= Sxr * r0[i] + Syr * r1[i];
}

// five consecutive image bytes starting at byte offset (sh/8) of the aligned word pair at `row`
__device__ __forceinline__ void load_row5(const uint8_t* row, int sh, float* f) {
  const uint32_t w0 = *reinterpret_cast<const uint32_t*>(row);
  const uint32_t w1 = *reinterpret_cast<const uint32_t*>(row + 4);
  const uint32_t lo = __funnelshift_r(w0, w1, sh);
  const uint32_t hi = w1 >> sh;
  f[0] = byte_to_float(lo, 0);
  f[1] = byte_to_float(lo, 1);
  f[2] = byte_to_float(lo, 2);
  f[3] = byte_to_float(lo, 3);
  f[4] = byte_to_float(hi, 0);
}
// seven consecutive bytes (reference image, global memory, read-only path)
__device__ __forceinline__ void load_row7(const uint8_t* row, int sh, float* g) {
  const uint32_t* wp = reinterpret_cast<const uint32_t*>(row);
  const uint32_t w0 = __ldg(wp), w1 = __ldg(wp + 1), w2 = __ldg(wp + 2);
  const uint32_t lo = __funnelshift_r(w0, w1, sh);
  const uint32_t hi = __funnelshift_r(w1, w2, sh);
  g[0] = byte_to_float(lo, 0);
  g[1] = byte_to_float(lo, 1);
  g[2] = byte_to_float(lo, 2);
  g[3] = byte_to_float(lo, 3);
  g[4] = byte_to_float(hi, 0);
  g[5] = byte_to_float(hi, 1);
  g[6] = byte_to_float(hi, 2);
}

// One patch of the residual pass.  weighted = point patch (:450-500: w = 1/(1+|r|), term = r*r*w); otherwise a
// segment sample (:612-637: unweighted sums, term = |r|).  Returns false if the warped patch is not fully
// inside the current image (isInFrame(halfsize)).
// Per-pixel values (bilinear intensity, residual, weight, chi2 term) are bit-identical to the reference's
// float arithmetic and are returned in t[16] (row-major, the reference's summation order); the five in-patch
// sums are accumulated per pixel in double from the exactly widened float operands, as the reference does
// for every pixel's J*J^T*w (:487-492).  PLSVO_FP32_SUMS builds the fp32-FMA variant for the A/B in
// profiles/ (0.4 % of pairs then terminate differently from the reference; tools/emulate_kernel_sums.py).
template <bool weighted, int NT>
__device__ __forceinline__ bool eval_patch(const uint8_t* __restrict__ img, int pitch, int cols, int rows,
                                           const float4* __restrict__ cache, int MP, int p, double u, double v,
                                           double* S /*[5]*/, float* __restrict__ tsc, float& tsum, f32x2 one2) {
  int ui, vi;
  float wTL, wTR, wBL, wBR;
  if (!patch_setup(u, v, cols, rows, 2, ui, vi, wTL, wTR, wBL, wBR)) return false;
  // 5x5 footprint, streamed row by row (two aligned 32-bit loads + funnel shift per row; rows are 4B-pitched).
  // The row loop is kept rolled: the pass loop must fit the 32 KB instruction cache.
  const int c0 = ui - 2;
  const int sh = (c0 & 3) * 8;
  const uint8_t* rowp = img + (size_t)(vi - 2) * pitch + (c0 & ~3);
  float ra[5], rb[5];
  load_row5(rowp, sh, ra);
#ifdef PLSVO_FP32_SUMS
  float Sxx = 0.f, Sxy = 0.f, Syy = 0.f, Sxr = 0.f, Syr = 0.f;
#else
  double Sxx = 0, Sxy = 0, Syy = 0, Sxr = 0, Syr = 0;
#endif
  float acc_f = 0.f;
  const float4* cp = cache + p;
#pragma unroll 1
  for (int y = 0; y < 4; ++y) {
    rowp += pitch;
    load_row5(rowp, sh, rb);
    const float4 ref4 = cp[0];
    const float4 dx4 = cp[4 * MP];
    const float4 dy4 = cp[8 * MP];
    cp += MP;
    const float refv[4] = {ref4.x, ref4.y, ref4.z, ref4.w};
    const float dxv[4] = {dx4.x, dx4.y, dx4.z, dx4.w};
    const float dyv[4] = {dy4.x, dy4.y, dy4.z, dy4.w};
#ifdef PLSVO_SCALAR_PIXELS
#pragma unroll
    for (int x = 0; x < 4; ++x) {
      const float cur = bilin(wTL, wTR, wBL, wBR, ra[x], ra[x + 1], rb[x], rb[x + 1]);
      const float res = __fsub_rn(cur, refv[x]);
      const float dx = dxv[x], dy = dyv[x];
      const float ares = fabsf(res);
      const float nw = weighted ? -weight_rcp(ares) : -1.0f;                           // :479 (negated)
      const float nterm = weighted ? __fmul_rn(__fmul_rn(res, res), nw) : -ares;       // :484 / :643 (negated)
#else
    // two pixels per instruction (FMUL2 / FADD2 / FFMA2); every operation is the reference's, rounded on its own
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int x0 = 2 * h;
      const f32x2 pa = pk2(ra[x0], ra[x0 + 1]), pb = pk2(ra[x0 + 1], ra[x0 + 2]);
      const f32x2 pc = pk2(rb[x0], rb[x0 + 1]), pd = pk2(rb[x0 + 1], rb[x0 + 2]);
      // ((wTL*a + wTR*b) + wBL*c) + wBR*d  (:458)
      f32x2 cur2 = add2_after_mul(mul2(pk2(wTL, wTL), pa), mul2(pk2(wTR, wTR), pb), one2);
      cur2 = add2_after_mul(cur2, mul2(pk2(wBL, wBL), pc), one2);
      cur2 = add2_after_mul(cur2, mul2(pk2(wBR, wBR), pd), one2);
      const f32x2 res2 = sub2(cur2, pk2(refv[x0], refv[x0 + 1]));
      float resv[2], nwv[2], ntv[2];
      upk2(res2, resv[0], resv[1]);
      if (weighted) {
        const f32x2 nw2 = neg_weight_rcp2(res2);                 // -1/(1+|r|)  (:479)
        const f32x2 nt2 = mul2(mul2(res2, res2), nw2);           // -(r*r*w)    (:484)
        upk2(nw2, nwv[0], nwv[1]);
        upk2(nt2, ntv[0], ntv[1]);
      } else {
        nwv[0] = nwv[1] = -1.0f;
        ntv[0] = -fabsf(resv[0]), ntv[1] = -fabsf(resv[1]);      // -|r|        (:643)
      }
#pragma unroll
      for (int xx = 0; xx < 2; ++xx) {
      const int x = x0 + xx;
      const float res = resv[xx], nw = nwv[xx], nterm = ntv[xx];
      const float dx = dxv[x], dy = dyv[x];
#endif
      // the scratch keeps the NEGATED term (its consumers subtract it): the sign costs nothing there, here it would
      tsc[(y * 4 + x) * NT] = nterm;
      acc_f = __fsub_rn(acc_f, nterm);
#ifdef PLSVO_FP32_SUMS
      const float wdx = weighted ? __fmul_rn(-nw, dx) : dx, wdy = weighted ? __fmul_rn(-nw, dy) : dy;
      Sxx = fmaf(wdx, dx, Sxx);
      Sxy = fmaf(wdx, dy, Sxy);
      Syy = fmaf(wdy, dy, Syy);
      Sxr = fmaf(wdx, res, Sxr);
      Syr = fmaf(wdy, res, Syr);
#else
      const double dxd = (double)dx, dyd = (double)dy, rd = (double)res;
      const double nwdx = weighted ? (double)nw * dxd : -dxd;  // exact products (24+24 bits), negated
      const double nwdy = weighted ? (double)nw * dyd : -dyd;
      Sxx = fma(-nwdx, dxd, Sxx);
      Sxy = fma(-nwdx, dyd, Sxy);
      Syy = fma(-nwdy, dyd, Syy);
      Sxr = fma(-nwdx, rd, Sxr);
      Syr = fma(-nwdy, rd, Syr);
#endif
#ifndef PLSVO_SCALAR_PIXELS
      }
#endif
    }
#pragma unroll
    for (int c = 0; c < 5; ++c) ra[c] = rb[c];
  }
  S[0] = (double)Sxx, S[1] = (double)Sxy, S[2] = (double)Syy, S[3] = (double)Sxr, S[4] = (double)Syr;
  tsum = acc_f;  // fl-sum of the 16 (positive) terms started from zero: the estimate of this patch's contribution
  return true;
}

// s <- fl(...fl(fl(s + t0) + t1)... + t15): the reference's float accumulator walking one patch whose terms sit
// in the thread's shared-memory scratch
template <int NT>
__device__ __forceinline__ float chain16(float s, const float* tsc) {
#pragma unroll
  for (int k = 0; k < 16; ++k) s = __fsub_rn(s, tsc[k * NT]);  // the scratch holds negated terms
  return s;
}
// the same walk from two starting values at once (even / odd mantissa at the bottom of a binade)
template <int NT>
__device__ __forceinline__ void chain16x2(float& s0, float& s1, const float* tsc) {
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    const float t = tsc[k * NT];  // negated term
    s0 = __fsub_rn(s0, t);
    s1 = __fsub_rn(s1, t);
  }
}

// Reference-patch precompute for one patch (:243-264 / :354-375): 16 interpolated intensities and
// central-difference gradients of the interpolated image, written as 12 float4 rows.
// V[a][b] = interpolated intensity at integer offset (a-1, b-1) from the patch origin; the reference
// evaluates the same bilinear expression for ref / dx / dy of neighbouring pixels (:251-258), so each
// value is computed once, in a rolled sliding window over the rows (V rows y, y+1, y+2 for pixel row y).
__device__ __forceinline__ void precompute_patch(const uint8_t* __restrict__ img, int pitch, int ui, int vi, float wTL,
                                                 float wTR, float wBL, float wBR, float4* __restrict__ cache, int MP,
                                                 int p) {
  const int c0 = ui - 3;
  const int sh = (c0 & 3) * 8;
  const uint8_t* rowp = img + (size_t)(vi - 3) * pitch + (c0 & ~3);
  float g0[7], g1[7], Va[6], Vb[6], Vc[6];
  load_row7(rowp, sh, g0);
  load_row7(rowp + pitch, sh, g1);
#pragma unroll
  for (int c = 0; c < 6; ++c) Va[c] = bilin(wTL, wTR, wBL, wBR, g0[c], g0[c + 1], g1[c], g1[c + 1]);
  rowp += 2 * pitch;
  load_row7(rowp, sh, g0);
#pragma unroll
  for (int c = 0; c < 6; ++c) Vb[c] = bilin(wTL, wTR, wBL, wBR, g1[c], g1[c + 1], g0[c], g0[c + 1]);
  // here g0 holds block row 2; loop invariant: g0 = block row y+2
  float4* cp = cache + p;
#pragma unroll 1
  for (int y = 0; y < 4; ++y) {
    rowp += pitch;
    load_row7(rowp, sh, g1);  // block row y+3
#pragma unroll
    for (int c = 0; c < 6; ++c) Vc[c] = bilin(wTL, wTR, wBL, wBR, g0[c], g0[c + 1], g1[c], g1[c + 1]);
    float refv[4], dxv[4], dyv[4];
#pragma unroll
    for (int x = 0; x < 4; ++x) {
      refv[x] = Vb[x + 1];
      dxv[x] = __fmul_rn(0.5f, __fsub_rn(Vb[x + 2], Vb[x]));
      dyv[x] = __fmul_rn(0.5f, __fsub_rn(Vc[x + 1], Va[x + 1]));
    }
    cp[0] = make_float4(refv[0], refv[1], refv[2], refv[3]);
    cp[4 * MP] = make_float4(dxv[0], dxv[1], dxv[2], dxv[3]);
    cp[8 * MP] = make_float4(dyv[0], dyv[1], dyv[2], dyv[3]);
    cp += MP;
#pragma unroll
    for (int c = 0; c < 6; ++c) Va[c] = Vb[c], Vb[c] = Vc[c];
#pragma unroll
    for (int c = 0; c < 7; ++c) g0[c] = g1[c];
  }
}

__device__ __forceinline__ void zero_gradients(float4* cache, int MP, int p) {
  const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int y = 0; y < 8; ++y) cache[(4 + y) * MP + p] = z;
}

// Thread 0, first half of one Gauss-Newton step of vk::NLLSSolver::optimizeGaussNewton: SparseImgAlign::solve()
// (:697-704) on the block totals and the candidate update T*exp(-x) (:709), formed while the walker warp is still
// chaining the chi2 items.  tot = [0..20]=H upper, [21..26]=Jres, [28]=n_meas, [29]=patches evaluated.
__device__ __noinline__ void gn_solve(PairCtl* ctl, const double* tot, int level) {
  ctl->n_meas_last = (long long)tot[28];
  ctl->patch_iters += (unsigned int)tot[29];
  ctl->iters_level[level] += 1;
  double xx[6];
  {
    double Hu[21], gg[6];
#pragma unroll
    for (int i = 0; i < 21; ++i) Hu[i] = tot[i];
#pragma unroll
    for (int i = 0; i < 6; ++i) gg[i] = tot[21 + i];
    if (!ldlt6_reg(Hu, gg, xx)) {
      // degenerate system: pivoted Eigen-style routine on the full symmetric matrix
      double* H = ctl->H_last;
      int idx = 0;
      for (int i = 0; i < 6; ++i)
        for (int j = i; j < 6; ++j) {
          H[i * 6 + j] = tot[idx];
          H[j * 6 + i] = tot[idx];
          ++idx;
        }
      for (int i = 0; i < 6; ++i) ctl->g[i] = tot[21 + i];
      ldlt6_solve(H, ctl->g, ctl->x, ctl->scratch);
#pragma unroll
      for (int i = 0; i < 6; ++i) xx[i] = ctl->x[i];
    }
  }
  if (isnan(xx[0])) ctl->stop = 1;
  double mx[6];
  double nm = 0.0;
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    mx[i] = -xx[i];
    nm = fmax(nm, fabs(xx[i]));
  }
  SE3q model;
  model.q.x = ctl->model[0], model.q.y = ctl->model[1], model.q.z = ctl->model[2], model.q.w = ctl->model[3];
  model.t = v3(ctl->model[4], ctl->model[5], ctl->model[6]);
  const SE3q cand = se3_mul(model, se3_exp(mx));
  se3_store(cand, ctl->cand);
  quat_to_R(cand.q, ctl->candR);
  ctl->cand_nm = nm;
}

// Thread 0, second half: the accept / rollback / convergence logic of vk::NLLSSolver::optimizeGaussNewton.
// chi2f is the pass's chi2 in the reference's summation order.
__device__ __noinline__ void gn_decide(PairCtl* ctl, const double* tot, float chi2f, int n_iter, double eps) {
  // chi2/n_meas_ : float / size_t -> float (:192)
  const double new_chi2 = (double)(chi2f / (float)(unsigned long long)ctl->n_meas_last);
  const bool reject = (ctl->iter > 0 && new_chi2 > ctl->chi2_prev) || ctl->stop;
  int flag;
  if (reject) {
    for (int i = 0; i < 7; ++i) ctl->model[i] = ctl->old_model[i];
    Quat q;
    q.x = ctl->model[0], q.y = ctl->model[1], q.z = ctl->model[2], q.w = ctl->model[3];
    quat_to_R(q, ctl->R);
    flag = 1;
  } else {
    for (int i = 0; i < 7; ++i) ctl->old_model[i] = ctl->model[i], ctl->model[i] = ctl->cand[i];
    for (int i = 0; i < 9; ++i) ctl->R[i] = ctl->candR[i];
    ctl->chi2_prev = new_chi2;
    flag = (ctl->cand_nm <= eps) ? 1 : 0;
  }
  ctl->t[0] = ctl->model[4], ctl->t[1] = ctl->model[5], ctl->t[2] = ctl->model[6];
  ctl->iter += 1;
  if (ctl->iter >= n_iter) flag = 1;
  if (flag) {  // last evaluated pass of this level: keep H_ (getFisherInformation, :97-102)
    int idx = 0;
    for (int i = 0; i < 6; ++i)
      for (int j = i; j < 6; ++j) {
        ctl->H_last[i * 6 + j] = tot[idx];
        ctl->H_last[j * 6 + i] = tot[idx];
        ++idx;
      }
  }
  ctl->flag = flag;
}

__device__ __forceinline__ void named_barrier_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
// producer side of a named barrier: counts this warp's threads in, does not wait
__device__ __forceinline__ void named_barrier_arrive(int id, int nthreads) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---- chi2 items (shared memory, 8 bytes): x = A_even (ulps added when the running sum's mantissa is even),
// y = [15:0] A_odd - A_even (signed) | [23:16] biased float exponent of the binade | [24] opaque | [31:25] opaque slot
__device__ __forceinline__ uint2 make_item(uint32_t Ae, uint32_t Ao, uint32_t ef, uint32_t opaque, uint32_t slot) {
  uint2 it;
  it.x = Ae;
  it.y = ((Ao - Ae) & 0xffffu) | (ef << 16) | (opaque << 24) | (slot << 25);
  return it;
}

// ---- level units: a pair's progress word and the state it carries between levels (global memory, L2) ----
__device__ __forceinline__ unsigned long long ld_acquire_gpu(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __noinline__ void unit_state_store(const PairCtl* ctl, AlignUnitState* s) {
  for (int i = 0; i < 7; ++i) s->model[i] = ctl->model[i];
  for (int i = 0; i < 9; ++i) s->R[i] = ctl->R[i];
  for (int i = 0; i < 3; ++i) s->t[i] = ctl->t[i];
  s->chi2_prev = ctl->chi2_prev;
  for (int i = 0; i < 36; ++i) s->H_last[i] = ctl->H_last[i];
  s->n_meas_last = ctl->n_meas_last;
  s->stop = ctl->stop, s->chi2_flags = ctl->chi2_flags;
  s->patch_iters = ctl->patch_iters, s->patch_levels = ctl->patch_levels;
  for (int l = 0; l < PLSVO_MAX_LEVELS; ++l) s->iters_level[l] = ctl->iters_level[l];
}
// L2 loads (ld.global.cg): the state was written by another SM
__device__ __noinline__ void unit_state_load(PairCtl* ctl, const AlignUnitState* s) {
  for (int i = 0; i < 7; ++i) ctl->model[i] = __ldcg(s->model + i);
  for (int i = 0; i < 9; ++i) ctl->R[i] = __ldcg(s->R + i);
  for (int i = 0; i < 3; ++i) ctl->t[i] = __ldcg(s->t + i);
  ctl->chi2_prev = __ldcg(&s->chi2_prev);
  for (int i = 0; i < 36; ++i) ctl->H_last[i] = __ldcg(s->H_last + i);
  ctl->n_meas_last = __ldcg(&s->n_meas_last);
  ctl->stop = __ldcg(&s->stop), ctl->chi2_flags = __ldcg(&s->chi2_flags);
  ctl->patch_iters = __ldcg(&s->patch_iters), ctl->patch_levels = __ldcg(&s->patch_levels);
  for (int l = 0; l < PLSVO_MAX_LEVELS; ++l) ctl->iters_level[l] = __ldcg(s->iters_level + l);
}

template <int NT, int MINB>
__global__ void __launch_bounds__(NT, MINB) sparse_img_align_kernel(const AlignArgs a) {
  constexpr int NW = NT / 32;
  constexpr int WALK = NW > 1 ? 1 : 0;  // warp that chains the chi2 items while thread 0 solves
  constexpr int SEGW = NW > 2 ? 2 : WALK;  // warp that sums the segments' chi2 terms meanwhile
  constexpr int kSerialThreads = 32 * (NW > 2 ? 3 : (NW > 1 ? 2 : 1));
  extern __shared__ __align__(128) unsigned char smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int MP = a.max_patches;
  const Layout L = make_layout(a.n_pts, a.n_segs, MP, a.max_seg_slots, a.smem_img_bytes, NT);
  PairCtl* ctl = reinterpret_cast<PairCtl*>(smem + L.ctl);
  double* red = reinterpret_cast<double*>(smem + L.red);
  double* tot = reinterpret_cast<double*>(smem + L.tot);
  double* chunk_tot = reinterpret_cast<double*>(smem + L.chunk_tot);
  uint2* items = reinterpret_cast<uint2*>(smem + L.items);
  int* item_cnt = reinterpret_cast<int*>(smem + L.cnt);
  float* opq = reinterpret_cast<float*>(smem + L.opq);
  uint8_t* seg_alive = smem + L.seg_alive;
  int* seg_N0 = reinterpret_cast<int*>(smem + L.seg_N0);
  int* seg_N = reinterpret_cast<int*>(smem + L.seg_N);
  int* seg_off = reinterpret_cast<int*>(smem + L.seg_off);
  int* seg_slot = reinterpret_cast<int*>(smem + L.seg_slot);
  uint16_t* slot_seg = reinterpret_cast<uint16_t*>(smem + L.slot_seg);
  const int max_slots = a.max_seg_slots;  // multiple of 32
  float* seg_term = reinterpret_cast<float*>(smem + L.seg_term);
  uint8_t* pt_vis = smem + L.pt_vis;
  uint8_t* img_s = smem + L.img;
  // per-CTA workspaces in global memory (L2 resident)
  float4* cache = a.ws_cache + (size_t)blockIdx.x * kCacheRows * MP;
  double* xyz = reinterpret_cast<double*>(smem + L.xyz);
  float* tsc = reinterpret_cast<float*>(smem + L.tsc) + tid;  // this thread's term k at tsc[k * NT]
  uint2* flat = reinterpret_cast<uint2*>(smem + L.flat);
  double* seg_px = a.ws_segpx + (size_t)blockIdx.x * 2 * a.max_seg_patches;  // 2-D centre of every segment sample
  const int RS = a.rec_cap * NT;                                     // record slots per component
  double* rec = a.ws_rec + (size_t)blockIdx.x * 5 * RS;               // five in-patch sums of this pass, per thread slot
  const f32x2 one2 = pk2(a.one, a.one);  // 1.0f from the host (see add2_after_mul)
  uint64_t* bar = reinterpret_cast<uint64_t*>(&ctl->mbar);
  if (tid == 0) {
    mbar_init(bar, 1);
    fence_mbarrier_init();
    fence_proxy_async();
  }
  __syncthreads();
  uint32_t bar_parity = 0;
  // Work queue.  Pair mode: ticket = pair.  Level units: ticket = (level index k, pair), k-major, so the unit of pair b at
  // level max_level - k is ticket k*B + b and the unit it continues from was handed out exactly B tickets earlier.
  for (;;) {
    __syncthreads();  // everyone is done with ctl of the previous pair
    if (tid == 0) {
      const int nb = (int)atomicAdd(a.work_counter, 1u);
      if (a.gate_chunk > 0 && nb < a.B) {
        // host-buffer pipeline: this pair's inputs are still in flight over PCIe until the copy stream
        // has bumped the arrival counter past its chunk
        const unsigned need = (unsigned)(nb / a.gate_chunk) + 1u;
        while (*reinterpret_cast<const volatile unsigned int*>(a.arrived) < need) __nanosleep(1000);
        __threadfence_system();
      }
      ctl->pair = nb;
      ctl->level_lo = a.level_units ? a.max_level - nb / a.B : a.min_level;
    }
    __syncthreads();
    const int ticket = ctl->pair;
    if (ticket >= a.B * (a.level_units ? a.max_level - a.min_level + 1 : 1)) break;
    const int unit = ticket / a.B;  // levels of this pair done before this unit
    const int b = ticket - unit * a.B;

    // feature counts are validated on upload; the clamp keeps a corrupted count from indexing out of bounds
    const int np = min(max(a.pt_count ? a.pt_count[b] : a.n_pts, 0), a.n_pts);
    const int ns = min(max(a.seg_count ? a.seg_count[b] : a.n_segs, 0), a.n_segs);
    const size_t po = (size_t)b * a.n_pts, so = (size_t)b * a.n_segs;

    if (np == 0 && ns == 0) {  // :58-62 early-out: return 0, cur pose untouched
      if (unit > 0) continue;  // the pair's first unit has written its outputs; nobody waits for an empty pair
      if (tid == 0) {
        for (int i = 0; i < 7; ++i) a.out_T[(size_t)b * 7 + i] = a.T_cur_w[(size_t)b * 7 + i];
        a.out_n_tracked[b] = 0;
        for (int i = 0; i < 36; ++i) a.out_H[(size_t)b * 36 + i] = 0.0;
        for (int l = 0; l < PLSVO_MAX_LEVELS; ++l) a.out_iters[(size_t)b * PLSVO_MAX_LEVELS + l] = 0;
        a.out_status[b] = 1;
        a.out_patch_iters[b] = 0;
        a.out_patch_levels[b] = 0;
      }
      for (int j = tid; j < a.n_segs; j += NT) a.out_seg_killed[so + j] = 0;
      continue;
    }

    if (tid == 0) {
      const SE3q T_ref = se3_load(a.T_ref_w + (size_t)b * 7);
      const SE3q T_ref_inv = se3_inverse(T_ref);
      se3_store(T_ref, ctl->T_ref);
      ctl->ref_pos[0] = T_ref_inv.t.x, ctl->ref_pos[1] = T_ref_inv.t.y, ctl->ref_pos[2] = T_ref_inv.t.z;
      ctl->n_opq = 0;
      if (unit == 0) {
        const SE3q T_cur = se3_load(a.T_cur_w + (size_t)b * 7);
        const SE3q model = se3_mul(T_cur, T_ref_inv);  // :80
        se3_store(model, ctl->model);
        quat_to_R(model.q, ctl->R);
        ctl->t[0] = model.t.x, ctl->t[1] = model.t.y, ctl->t[2] = model.t.z;
        ctl->chi2_prev = 1e10;
        ctl->stop = 0;
        ctl->n_meas_last = 0;
        ctl->patch_iters = 0;
        ctl->patch_levels = 0;
        ctl->chi2_flags = 0;
        for (int i = 0; i < 36; ++i) ctl->H_last[i] = 0.0;
        for (int l = 0; l < PLSVO_MAX_LEVELS; ++l) ctl->iters_level[l] = 0;
      }
    }
    // Host-buffer pipeline with lean inputs: pyramid levels above a.derive_from were not shipped; this CTA forms them
    // for its own pair by vk::halfSample (truncating 2x2 mean, frame_utils::createImgPyramid, src/frame.cpp:171-180)
    // right where the pair's finest level has just landed.  (A separate pyramid kernel could not become resident next
    // to the persistent grid that is waiting for it.)
    if (a.derive_from >= 0) {
      for (int l = a.derive_from + 1; l <= a.max_level; ++l) {
        const int cols = a.width >> l, rows = a.height >> l;
        const int pin = (int)a.pitch[l - 1], pout = (int)a.pitch[l];
#pragma unroll 1
        for (int which = 0; which < 2; ++which) {
          const uint8_t* src = (which ? a.cur_img[l - 1] : a.ref_img[l - 1]) + (size_t)b * a.stride[l - 1];
          uint8_t* dst = const_cast<uint8_t*>(which ? a.cur_img[l] : a.ref_img[l]) + (size_t)b * a.stride[l];
          for (int y = warp; y < rows; y += NW) {
            const uint8_t* r0 = src + (size_t)(2 * y) * pin;
            for (int x = lane; x < cols; x += 32)
              dst[(size_t)y * pout + x] = (uint8_t)(((int)r0[2 * x] + (int)r0[2 * x + 1] + (int)r0[pin + 2 * x] + (int)r0[pin + 2 * x + 1]) >> 2);
          }
        }
        __syncthreads();  // level l is the source of level l+1
      }
      asm volatile("fence.proxy.async;" ::: "memory");  // the bulk copies of the level loop read what was written here
      __syncthreads();
    }
    __syncthreads();
    const double rpx = ctl->ref_pos[0], rpy = ctl->ref_pos[1], rpz = ctl->ref_pos[2];

    // per-pair point setup: xyz_ref = f * |pos - ref_pos| (:229-230), kept as (X/Z, Y/Z, 1/Z); visibility cleared
    for (int i = tid; i < np; i += NT) {
      pt_vis[i] = 0;
      double fd[3];
      const double* f = fd;
      if (a.pt_f) f = a.pt_f + (po + i) * 3;
      else cam2world(a, a.pt_px + (po + i) * 2, fd);  // bearing not shipped: PointFeat's own construction (feature.cpp:42)
      double depth;
      if (a.pt_depth) {
        depth = a.pt_depth[po + i];
      } else {
        const double* pos = a.pt_pos + (po + i) * 3;
        const double dx = pos[0] - rpx, dy = pos[1] - rpy, dz = pos[2] - rpz;
        depth = sqrt(dx * dx + dy * dy + dz * dz);
      }
      const double zi = 1.0 / (f[2] * depth);  // z_inv of Frame::jacobian_xyz2uv (frame.h:144), constant per pair
      xyz[0 * MP + i] = (f[0] * depth) * zi;
      xyz[1 * MP + i] = (f[1] * depth) * zi;
      xyz[2 * MP + i] = zi;
    }
    for (int j = tid; j < ns; j += NT) {
      seg_alive[j] = a.seg_valid ? (a.seg_valid[so + j] ? 1 : 0) : 1;
      seg_N0[j] = seg_num_samples0(a.seg_spx + (so + j) * 2, a.seg_epx + (so + j) * 2, a.seg_length[so + j]);
    }
    if (unit > 0) {
      const unsigned char* ust = a.unit_state + (size_t)b * a.unit_state_stride;
      // Continue the pair where the unit of the level above left it.  No deadlock: that unit holds ticket - B, which was
      // handed out before this one, so a resident CTA is running it; and it only ever waits for a ticket earlier still.
      if (tid == 0) {
        const unsigned long long want = (a.unit_epoch << 4) | (unsigned long long)unit;
        while (ld_acquire_gpu(a.unit_done + b) != want) __nanosleep(256);
        unit_state_load(ctl, reinterpret_cast<const AlignUnitState*>(ust));
      }
      __syncthreads();
      const unsigned char* vis = ust + sizeof(AlignUnitState);
      for (int i = tid; i < np; i += NT) pt_vis[i] = __ldcg(vis + i);
      for (int j = tid; j < ns; j += NT) seg_alive[j] = __ldcg(vis + a.n_pts + j);
    }
    unsigned int my_patch_levels = 0;
    const int n_chunks = (np + 31) >> 5;       // 32-patch chunks of the point list
    const int rounds = (np + NT - 1) / NT;     // rounds of NT point patches per pass

    for (int level = a.level_units ? ctl->level_lo : a.max_level; level >= ctl->level_lo; --level) {
      const int cols = a.width >> level, rows = a.height >> level;
      const int pitch = (int)a.pitch[level];
      const float scale = 1.0f / (float)(1 << level);
      const double dscale = (double)scale;
      const uint8_t* ref_img = a.ref_img[level] + (size_t)b * a.stride[level];
      const uint8_t* cur_img_g = a.cur_img[level] + (size_t)b * a.stride[level];
      const bool stage = a.img_in_smem[level] != 0;
      const uint8_t* cur_img = stage ? img_s : cur_img_g;
      __syncthreads();  // previous level's readers of img_s are done
      if (tid == 0) {
        if (stage) {
          const uint32_t bytes = (uint32_t)rows * (uint32_t)pitch;
          fence_proxy_async();
          mbar_expect_tx(bar, bytes);
          bulk_g2s(img_s, cur_img_g, bytes, bar);
        }
        ctl->iter = 0;
        for (int i = 0; i < 7; ++i) ctl->old_model[i] = ctl->model[i];
      }
      // ---- segment sampling at this level (:285-332) ----
      for (int j = tid; j < ns; j += NT) {
        int N = 0;
        if (seg_alive[j]) {
          const double* spx = a.seg_spx + (so + j) * 2;
          const double* epx = a.seg_epx + (so + j) * 2;
          const int sx = (int)(spx[0] * dscale), sy = (int)(spx[1] * dscale);
          const int ex = (int)(epx[0] * dscale), ey = (int)(epx[1] * dscale);
          if (cam_in_frame(sx, sy, 3, level, a.width, a.height) && cam_in_frame(ex, ey, 3, level, a.width, a.height))
            N = 1 + ((seg_N0[j] - 1) >> level);
        }
        seg_N[j] = N;
        seg_term[j] = 0.f;
      }
      for (int q = tid; q < max_slots; q += NT) slot_seg[q] = 0xffffu;
      __syncthreads();
      if (warp == 0) {  // exclusive scan of seg_N -> seg_off (cache offsets in patches, :282-292) + lane groups
        int carry = 0;
        for (int base = 0; base < ns; base += 32) {
          const int j = base + lane;
          const int v = (j < ns) ? seg_N[j] : 0;
          int incl = v;
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) {
            const int n = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += n;
          }
          if (j < ns) seg_off[j] = carry + incl - v;
          carry += __shfl_sync(0xffffffffu, incl, 31);
        }
        // Lane groups: segment j gets 2^k consecutive lanes, 2^k = smallest power of two >= min(N_j, 32).
        // Groups are laid out class by class, largest first, so every group is aligned to its own size
        // and never straddles a warp.
        int slot_base = 0;
        for (int cls = 5; cls >= 0; --cls) {
          int cnt = 0;
          for (int base = 0; base < ns; base += 32) {
            const int j = base + lane;
            const int N = (j < ns) ? seg_N[j] : 0;
            int k = -1;
            if (N > 0) {
              k = 0;
              while ((1 << k) < N && k < 5) ++k;
            }
            const unsigned m = __ballot_sync(0xffffffffu, k == cls);
            if (k == cls) seg_slot[j] = slot_base + ((cnt + __popc(m & ((1u << lane) - 1u))) << cls);
            cnt += __popc(m);
          }
          slot_base += cnt << cls;
        }
        if (lane == 0) {
          ctl->n_seg_patches = carry;
          ctl->n_seg_slots = slot_base;
        }
      }
      __syncthreads();
      const int n_sp = min(ctl->n_seg_patches, a.max_seg_patches);
      const int n_patches = np + n_sp;
      const int n_seg_slots = min((ctl->n_seg_slots + 31) & ~31, max_slots);
      // ---- expand segments into sample patches: 2D centre and 3D point by repeated addition (:323-335) ----
      for (int j = tid; j < ns; j += NT) {
        const int N = seg_N[j];
        if (N == 0) continue;
        const double* spx = a.seg_spx + (so + j) * 2;
        const double* epx = a.seg_epx + (so + j) * 2;
        const double dif[2] = {epx[0] - spx[0], epx[1] - spx[1]};
        const double nm1 = (double)(unsigned long long)(N - 1);
        const double inc2d0 = dif[0] * dscale / nm1, inc2d1 = dif[1] * dscale / nm1;
        double px0 = spx[0] * dscale, px1 = spx[1] * dscale;
        double sfd[3], efd[3];
        const double *sf = sfd, *ef = efd;
        if (a.seg_sf) sf = a.seg_sf + (so + j) * 3;
        else cam2world(a, spx, sfd);  // LineFeat's own construction (feature.cpp:98-99)
        if (a.seg_ef) ef = a.seg_ef + (so + j) * 3;
        else cam2world(a, epx, efd);
        double p_depth, q_depth;
        if (a.seg_sdepth) {
          p_depth = a.seg_sdepth[so + j];
        } else {
          const double* sp = a.seg_spos + (so + j) * 3;
          const double d0 = sp[0] - rpx, d1 = sp[1] - rpy, d2 = sp[2] - rpz;
          p_depth = sqrt(d0 * d0 + d1 * d1 + d2 * d2);
        }
        if (a.seg_edepth) {
          q_depth = a.seg_edepth[so + j];
        } else {
          const double* ep = a.seg_epos + (so + j) * 3;
          const double d0 = ep[0] - rpx, d1 = ep[1] - rpy, d2 = ep[2] - rpz;
          q_depth = sqrt(d0 * d0 + d1 * d1 + d2 * d2);
        }
        const double P0 = sf[0] * p_depth, P1 = sf[1] * p_depth, P2 = sf[2] * p_depth;
        const double Q0 = ef[0] * q_depth, Q1 = ef[1] * q_depth, Q2 = ef[2] * q_depth;
        const double i0 = (Q0 - P0) / nm1, i1 = (Q1 - P1) / nm1, i2 = (Q2 - P2) / nm1;
        double X = P0, Y = P1, Z = P2;
        const int off = seg_off[j];
        {
          int g = 1;
          while (g < N && g < 32) g <<= 1;
          const int s0 = seg_slot[j];
          for (int n = 0; n < g; ++n)
            if (s0 + n < max_slots) slot_seg[s0 + n] = (uint16_t)j;
        }
        for (int n = 0; n < N; ++n) {
          const int sp_idx = off + n;
          if (sp_idx < n_sp) {
            seg_px[2 * sp_idx] = px0;
            seg_px[2 * sp_idx + 1] = px1;
            const double zi = 1.0 / Z;
            xyz[0 * MP + np + sp_idx] = X * zi;
            xyz[1 * MP + np + sp_idx] = Y * zi;
            xyz[2 * MP + np + sp_idx] = zi;
          }
          px0 += inc2d0, px1 += inc2d1;
          X += i0, Y += i1, Z += i2;
        }
      }
      __syncthreads();
      // ---- reference patch cache (:195-378) ----
      for (int p = tid; p < n_patches; p += NT) {
        double u, v;
        const bool is_pt = p < np;
        if (is_pt) {
          if (a.pt_valid && !a.pt_valid[po + p]) continue;
          const double* px = a.pt_px + (po + p) * 2;
          u = px[0] * dscale, v = px[1] * dscale;
        } else {
          u = seg_px[2 * (p - np)], v = seg_px[2 * (p - np) + 1];
        }
        int ui, vi;
        float wTL, wTR, wBL, wBR;
        const bool in = patch_setup(u, v, cols, rows, 3, ui, vi, wTL, wTR, wBL, wBR);
        if (!in) {
          // points: skipped at this level (:218-219); their Jacobian columns were zeroed (:85).
          // segment samples are inside by construction; guard only protects against malformed input.
          if (!is_pt || pt_vis[p]) zero_gradients(cache, MP, p);
          continue;
        }
        if (is_pt) pt_vis[p] = 1;
        precompute_patch(ref_img, pitch, ui, vi, wTL, wTR, wBL, wBR, cache, MP, p);
        ++my_patch_levels;
      }
      if (stage) {
        mbar_wait(bar, bar_parity);
        bar_parity ^= 1u;
      }
      __syncthreads();

      // ---- Gauss-Newton iterations at this level (vk::NLLSSolver::optimizeGaussNewton) ----
      const double cJ = fabs(a.fx) / (double)(1 << level);  // focal_length / 2^level (:262)
      const double cJ2 = cJ * cJ;
      for (;;) {
        const double R0 = ctl->R[0], R1 = ctl->R[1], R2 = ctl->R[2], R3 = ctl->R[3], R4 = ctl->R[4], R5 = ctl->R[5],
                     R6 = ctl->R[6], R7 = ctl->R[7], R8 = ctl->R[8];
        const double t0 = ctl->t[0], t1 = ctl->t[1], t2 = ctl->t[2];
        int n_meas_acc = 0, n_patch_acc = 0;
#ifdef PLSVO_TREE_CHI2
        double chi2_tree = 0.0;
#endif
        // this thread's 21 (upper-triangular H) + 6 (Jres) accumulators of the pass
        double acc[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) acc[i] = 0.0;
        double prefix_rounds = 0.0;  // estimate of the float chi2 accumulator after all earlier rounds
        // ======== point patches (:380-502), one round of NT consecutive patches at a time ========
        for (int r = 0; r < rounds; ++r) {
          const int c = r * NW + warp;  // 32-patch chunk of this warp: patches [32c, 32c+32) in list order
          const int p = c * 32 + lane;
          float Tf = 0.f;
          bool ok = false;
          if (p < np && pt_vis[p]) {
            const double xn = xyz[0 * MP + p], yn = xyz[1 * MP + p], zi = xyz[2 * MP + p];
            const double xc = R0 * xn + R1 * yn + (R2 + t0 * zi);  // (R*xyz_ref + t) / Z_ref
            const double yc = R3 * xn + R4 * yn + (R5 + t1 * zi);
            const double zc = R6 * xn + R7 * yn + (R8 + t2 * zi);
            const double izc = __drcp_rn(zc);
            const double u = (a.fx * (xc * izc) + a.cx) * dscale;  // world2cam(xyz)*scale (:425)
            const double v = (a.fy * (yc * izc) + a.cy) * dscale;
            double S[5];
            ok = eval_patch<true, NT>(cur_img, pitch, cols, rows, cache, MP, p, u, v, S, tsc, Tf, one2);
            if (ok) {
              // normal equations: rank-2 update with the two projection-Jacobian rows of the patch
              rank2_update(acc, xn, yn, zi, S[0] * cJ2, S[1] * cJ2, S[2] * cJ2, S[3] * cJ, S[4] * cJ);
              n_meas_acc += 16;
              n_patch_acc += 1;
            }
          }
          if (!ok) Tf = 0.f;  // not evaluated: contributes nothing (its scratch terms are stale and never read)
#ifdef PLSVO_TREE_CHI2
          chi2_tree += (double)Tf;
#else
          if (c >= n_chunks) {
            // a warp whose chunk lies beyond the point list (last round only) signals the round barrier without waiting
            // and goes on to its segment rounds: it needs none of the totals the others are about to exchange
            named_barrier_arrive(2, NT);
            continue;
          }
          // -- estimate of the accumulator before this patch: exact prefix sum of the patch totals --
          double incl = (double)Tf;
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) {
            const double n = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += n;
          }
          if (lane == 31) chunk_tot[c] = incl;
          named_barrier_sync(2, NT);  // every chunk total of this round is published (empty chunks only arrive)
          double P = prefix_rounds;
#pragma unroll
          for (int w = 0; w < NW; ++w) {
            const double tw = (r * NW + w < n_chunks) ? chunk_tot[r * NW + w] : 0.0;
            if (w < warp) P += tw;
            prefix_rounds += tw;
          }
          P += incl - (double)Tf;
          if (c < n_chunks) {
            // -- classify: the float accumulator s_in before this patch satisfies |s_in - P| <= delta*P and the one
            // after it |s_out - (P+T)| <= delta*(P+T), delta = (#terms so far)*2^-24 (+ the estimate's own error) --
            const double delta = (double)(16 * (p + 2)) * 6.0e-8 + 2.0e-6;
            const double lo = P * (1.0 - delta), hi = (P + (double)Tf) * (1.0 + delta);
            const int e_lo = (__double2hiint(lo) >> 20) - 1023, e_hi = (__double2hiint(hi) >> 20) - 1023;
            uint32_t ef = 0, opaque = 0, Ae = 0, Ao = 0, slot = 0;
            if (!ok) {
              // no terms: identity map.  It joins the binade of the estimate so that it merges with its neighbours
              // (P == 0: still in front of the first non-zero term).
              if (P != 0.0 && e_lo == e_hi && e_lo >= -100 && e_lo <= 100) ef = (uint32_t)(e_lo + 127);
              else if (P != 0.0) ef = 255u;  // next to a power of two: a group of its own, still the identity
            } else if (P == 0.0) {
              opaque = (Tf != 0.f) ? 1u : 0u;  // leading zeros leave the accumulator at 0
            } else if (e_lo != e_hi || e_lo < -100 || e_lo > 100) {
              opaque = 1u;
            } else {
              // inside binade e: the 16 additions add A[parity of s_in's mantissa] ulps
              ef = (uint32_t)(e_lo + 127);
              const uint32_t b0 = ef << 23;
              float s0 = __uint_as_float(b0), s1 = __uint_as_float(b0 | 1u);
              chain16x2<NT>(s0, s1, tsc);
              Ae = __float_as_uint(s0) - b0;
              Ao = __float_as_uint(s1) - (b0 | 1u);
            }
            if (opaque) {
              const int idx = atomicAdd(&ctl->n_opq, 1);
              if (idx < kOpqCap) {
                slot = (uint32_t)idx;
#pragma unroll
                for (int k = 0; k < 16; ++k) opq[idx * 16 + k] = tsc[k * NT];
              } else {
                atomicOr(&ctl->chi2_flags, 1);
                opaque = 0u;  // dropped from the exact chain; the walker falls back to the estimate
              }
            }
            // -- compose the maps of consecutive patches of the same binade (segmented inclusive scan) --
            const uint32_t ef_prev = __shfl_up_sync(0xffffffffu, ef, 1);
            const uint32_t op_prev = __shfl_up_sync(0xffffffffu, opaque, 1);
            uint32_t head = (lane == 0 || opaque || op_prev || ef != ef_prev) ? 1u : 0u;
            const uint32_t heads = __ballot_sync(0xffffffffu, head);
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
              const uint32_t pAe = __shfl_up_sync(0xffffffffu, Ae, d);
              const uint32_t pAo = __shfl_up_sync(0xffffffffu, Ao, d);
              const uint32_t phead = __shfl_up_sync(0xffffffffu, head, d);
              if (lane >= d && !head) {
                // earlier map first: parity p -> p ^ (A_prev[p] & 1), then this lane's map
                const uint32_t nAe = pAe + ((pAe & 1u) ? Ao : Ae);
                const uint32_t nAo = pAo + ((pAo & 1u) ? Ae : Ao);
                Ae = nAe, Ao = nAo;
                head = phead;
              }
            }
            const bool tail = lane == 31 || ((heads >> (lane + 1)) & 1u);
            const uint32_t tails = __ballot_sync(0xffffffffu, tail);
            if (tail) items[c * 32 + __popc(tails & ((1u << lane) - 1u))] = make_item(Ae, Ao, ef, opaque, slot);
            if (lane == 0) item_cnt[c] = __popc(tails);
          }
#endif
        }
        // ======== segment samples (:504-695).  Every segment owns a group of G = 2^k consecutive lanes of one warp
        // (G >= its sample count, or the whole warp looping over samples), so the per-segment gate / weight
        // (:640-688) is a few shuffles: no block barrier.  Warps take segment rounds from the top so they interleave
        // with the point rounds. ========
        for (int base = (NW - 1 - warp) * 32; base < n_seg_slots; base += NT) {
          const int q = base + lane;
          const int j = slot_seg[q];
          const bool has = j < ns;
          const bool seg_ok = has && seg_alive[j];
          const int Ns = has ? seg_N[j] : 0;  // lane-group structure of the level (fixed for all its passes)
          const int N = seg_ok ? Ns : 0;      // samples to evaluate in this pass
          const int off = has ? seg_off[j] : 0;
          const int n0 = has ? q - seg_slot[j] : 0;
          int G = 1;
          while (G < Ns && G < 32) G <<= 1;
          const int gbase = lane - n0;  // first lane of this lane's group
          int trips = seg_ok ? (Ns + G - 1) / G : 0, gmax = seg_ok ? G : 0;
#pragma unroll
          for (int d = 16; d >= 1; d >>= 1) {
            trips = max(trips, __shfl_xor_sync(0xffffffffu, trips, d));
            gmax = max(gmax, __shfl_xor_sync(0xffffffffu, gmax, d));
          }
          float s_tok = 0.f;  // the reference's res_ accumulator (:643-646) handed from sample to sample
          int first_bad = 0x7fffffff;
          unsigned ok_trips = 0u;  // bit t: this lane's sample of trip t was evaluated
          double S[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
          int p = 0;
          for (int trip = 0; trip < trips; ++trip) {
            const int n = n0 + trip * G;
            const bool active = n < N;
            float Tf = 0.f;
            bool ok = false;
            if (active) {
              p = np + off + n;
              const double xn = xyz[0 * MP + p], yn = xyz[1 * MP + p], zi = xyz[2 * MP + p];
              const double xc = R0 * xn + R1 * yn + (R2 + t0 * zi);
              const double yc = R3 * xn + R4 * yn + (R5 + t1 * zi);
              const double zc = R6 * xn + R7 * yn + (R8 + t2 * zi);
              const double izc = __drcp_rn(zc);
              const double u = (a.fx * (xc * izc) + a.cx) * dscale;
              const double v = (a.fy * (yc * izc) + a.cy) * dscale;
              ok = eval_patch<false, NT>(cur_img, pitch, cols, rows, cache, MP, p, u, v, S, tsc, Tf, one2);
              if (ok) {
                ok_trips |= 1u << (trip & 31);
                if (trips > 1) {  // segment longer than a warp: park the sums until its weight is known
                  if (trip < a.rec_cap) {
                    double* rp = rec + trip * NT + tid;
#pragma unroll
                    for (int k = 0; k < 5; ++k) rp[k * RS] = S[k];
                  } else {
                    atomicOr(&ctl->chi2_flags, 4);  // host plan violated (never)
                  }
                }
              } else {
                first_bad = min(first_bad, n);
              }
            }
            // res_ += fabsf(res) over the samples in order, 16 pixels each (:643-646): the accumulator walks the
            // group's lanes; a lane without an evaluated sample hands it on unchanged
            for (int g = 0; g < gmax; ++g) {
              const float prev = __shfl_sync(0xffffffffu, s_tok, gbase + ((n0 - 1) & (G - 1)));
              if (n0 == g) {
                const float s_in = (g == 0 && trip == 0) ? 0.f : prev;
                s_tok = (active && ok) ? (s_in == 0.f ? Tf : chain16<NT>(s_in, tsc)) : s_in;
              }
            }
          }
          // group results: the accumulator sits on the group's last lane; first failing sample by xor tree
          float res_ = __shfl_sync(0xffffffffu, s_tok, gbase + G - 1);
#pragma unroll
          for (int d = 16; d >= 1; d >>= 1) {
            const int fb = __shfl_xor_sync(0xffffffffu, first_bad, d);
            if (d < G) first_bad = min(first_bad, fb);
          }
          double sH = 0.0, sJ = 0.0;
          if (N > 0 && n0 == 0) {  // the group's first lane settles the segment
            const bool good = first_bad >= N;
            n_patch_acc += good ? N : first_bad;  // samples evaluated before the loop stops (:588-594)
            res_ = (float)((double)res_ / (double)(unsigned long long)N);  // :647
            if (good && (double)res_ < 200.0) {
              const float w = (float)(1.0 / (1.0 + (double)res_));  // :675
              sH = (double)w / (double)res_ * cJ2;                  // H += H_*weight/res_ (:681)
              sJ = (double)w * cJ;                                  // Jres += Jres_*weight (:682)
              seg_term[j] = __fmul_rn(__fmul_rn(res_, res_), w);    // chi2 += res_*res_*weight (:683)
#ifdef PLSVO_TREE_CHI2
              chi2_tree += (double)seg_term[j];
#endif
              n_meas_acc += 1;                                      // :684
            } else {
              seg_term[j] = 0.f;
              seg_alive[j] = 0;  // it->feat3D = NULL (:688); the group's lanes have all read it already
            }
          }
          sH = __shfl_sync(0xffffffffu, sH, gbase);  // the segment's weight to all lanes of its group
          sJ = __shfl_sync(0xffffffffu, sJ, gbase);
          if (sH != 0.0 || sJ != 0.0) {  // accepted segment: its samples enter the normal equations
            if (trips == 1) {
              if (ok_trips) rank2_update(acc, xyz[0 * MP + p], xyz[1 * MP + p], xyz[2 * MP + p], S[0] * sH, S[1] * sH, S[2] * sH,
                                         S[3] * sJ, S[4] * sJ);
            } else {
              for (int trip = 0; trip < trips && trip < a.rec_cap; ++trip) {
                if (!((ok_trips >> (trip & 31)) & 1u)) continue;
                const int pp = np + off + n0 + trip * G;
                const double* rp = rec + trip * NT + tid;
                rank2_update(acc, xyz[0 * MP + pp], xyz[1 * MP + pp], xyz[2 * MP + pp], rp[0] * sH, rp[RS] * sH, rp[2 * RS] * sH,
                             rp[3 * RS] * sJ, rp[4 * RS] * sJ);
              }
            }
          }
        }
        acc[28] = (double)n_meas_acc;
        acc[29] = (double)n_patch_acc;
#ifdef PLSVO_TREE_CHI2
        acc[27] = chi2_tree;  // (variant for the A/B only) chi2 by tree sum, not in the reference's order
#endif
        // ---- block reduction (deterministic order) ----
        const double mine = warp_reduce32(acc, lane);
        red[warp * 32 + lane] = mine;
        __syncthreads();
        if (warp == 0) {
          double s = 0.0;
#pragma unroll
          for (int w = 0; w < NW; ++w) s += red[w * 32 + lane];
          tot[lane] = s;
          __syncwarp();
          if (lane == 0) gn_solve(ctl, tot, level);
        }
#ifdef PLSVO_TREE_CHI2
        if (warp == WALK && lane == 0) ctl->chi2f = 0.f;
        if (false) {
#else
        if (warp == WALK) {
#endif
          // ---- chi2 in the reference's order: chain the composed maps and the opaque patches ----
          float s = 0.f;
          uint32_t bad = 0;
          for (int c = 0; c < n_chunks;) {
            // gather the items of the next chunks (as many as fit 64 entries) into one list, in list order
            const int cc = c + lane;
            const int my_cnt = (cc < n_chunks) ? item_cnt[cc] : 0;
            int incl = my_cnt;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
              const int n = __shfl_up_sync(0xffffffffu, incl, d);
              if (lane >= d) incl += n;
            }
            const int nfit = max(1, __popc(__ballot_sync(0xffffffffu, cc < n_chunks && incl <= 64)));
            for (int j = 0; j < nfit; ++j) {
              const int cnt_j = __shfl_sync(0xffffffffu, my_cnt, j), off_j = __shfl_sync(0xffffffffu, incl - my_cnt, j);
              if (lane < cnt_j) flat[off_j + lane] = items[(c + j) * 32 + lane];
            }
            const int total = __shfl_sync(0xffffffffu, incl, nfit - 1);
            __syncwarp();
            for (int b0 = 0; b0 < total; b0 += 32) {
              uint2 it = make_uint2(0u, 0u);
              if (b0 + lane < total) it = flat[b0 + lane];
              float4 q0 = make_float4(0.f, 0.f, 0.f, 0.f), q1 = q0, q2 = q0, q3 = q0;
              if ((it.y >> 24) & 1u) {  // this lane's item is an opaque patch: fetch its 16 terms now, off the chain
                const float4* o4 = reinterpret_cast<const float4*>(opq + (it.y >> 25) * 16);
                q0 = o4[0], q1 = o4[1], q2 = o4[2], q3 = o4[3];
              }
              const float tr[16] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x, q2.y, q2.z, q2.w, q3.x, q3.y, q3.z, q3.w};
              const int m = min(32, total - b0);
              for (int k = 0; k < m; ++k) {
                const uint32_t ix = __shfl_sync(0xffffffffu, it.x, k), iy = __shfl_sync(0xffffffffu, it.y, k);
                if ((iy >> 24) & 1u) {
                  // opaque patch: its owner lane adds the 16 terms to the (warp-uniform) accumulator, then everyone
                  // takes the owner's result
                  float so = s;
#pragma unroll
                  for (int i = 0; i < 16; ++i) so = __fsub_rn(so, tr[i]);  // negated terms
                  s = __shfl_sync(0xffffffffu, so, k);
                } else {
                  const uint32_t dA = (uint32_t)(int)(short)(iy & 0xffffu);
                  if (ix | dA) {  // not the identity
                    uint32_t bits = __float_as_uint(s);
                    bad |= (bits >> 23) ^ ((iy >> 16) & 0xffu);
                    bits += (bits & 1u) ? ix + dA : ix;
                    s = __uint_as_float(bits);
                  }
                }
              }
            }
            __syncwarp();
            c += nfit;
          }
          if (lane == 0) {
            if (ctl->n_opq > kOpqCap) {
              // opaque buffer overflowed (flag 1): fall back to the estimate of the point sum for this pass
              double e = 0.0;
              for (int c = 0; c < n_chunks; ++c) e += chunk_tot[c];
              s = (float)e;
            }
            if (bad) atomicOr(&ctl->chi2_flags, 2);
            ctl->chi2f = s;  // pt_chi2 (:484); seg_chi2 is added by the decision (:171)
            ctl->n_opq = 0;
          }
        }
        if (warp == SEGW) {
          float s2 = 0.f;  // seg_chi2 (:683): one term per accepted segment, in list order (others hold +0, a no-op)
#pragma unroll 8
          for (int j = 0; j < ns; ++j) s2 = __fadd_rn(s2, seg_term[j]);
          if (lane == 0) ctl->seg_chi2f = s2;
        }
        // chi2 (walker warp, segment warp) -> decision (thread 0); the warps arrive converged: a named barrier counts
        // whole warps
        if (NW > 1 && warp * 32 < kSerialThreads) named_barrier_sync(1, kSerialThreads);
#ifdef PLSVO_TREE_CHI2
        if (tid == 0) gn_decide(ctl, tot, (float)tot[27], a.n_iter, a.eps);
#else
        if (tid == 0) gn_decide(ctl, tot, __fadd_rn(ctl->chi2f, ctl->seg_chi2f), a.n_iter, a.eps);  // pt_chi2 + seg_chi2 (:171)
#endif
        __syncthreads();
        if (ctl->flag) break;
      }
    }  // levels

    // ---- results ----
    {
      unsigned int v = my_patch_levels;
#pragma unroll
      for (int d = 16; d >= 1; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
      if (lane == 0 && v) atomicAdd(&ctl->patch_levels, v);
    }
    if (ctl->level_lo > a.min_level) {  // hand the pair on to its unit at the next finer level
      unsigned char* ust = a.unit_state + (size_t)b * a.unit_state_stride;
      unsigned char* vis = ust + sizeof(AlignUnitState);
      for (int i = tid; i < np; i += NT) vis[i] = pt_vis[i];
      for (int j = tid; j < ns; j += NT) vis[a.n_pts + j] = seg_alive[j];
      __syncthreads();
      if (tid == 0) {
        unit_state_store(ctl, reinterpret_cast<AlignUnitState*>(ust));
        __threadfence();
        st_release_gpu(a.unit_done + b, (a.unit_epoch << 4) | (unsigned long long)(a.max_level - ctl->level_lo + 1));
      }
      continue;
    }
    for (int j = tid; j < a.n_segs; j += NT) {
      const bool valid0 = (j < ns) && (a.seg_valid ? a.seg_valid[so + j] != 0 : true);
      a.out_seg_killed[so + j] = (valid0 && !seg_alive[j]) ? 1 : 0;
    }
    __syncthreads();
    if (tid == 0) {
      SE3q model, T_ref;
      model.q.x = ctl->model[0], model.q.y = ctl->model[1], model.q.z = ctl->model[2], model.q.w = ctl->model[3];
      model.t = v3(ctl->model[4], ctl->model[5], ctl->model[6]);
      T_ref.q.x = ctl->T_ref[0], T_ref.q.y = ctl->T_ref[1], T_ref.q.z = ctl->T_ref[2], T_ref.q.w = ctl->T_ref[3];
      T_ref.t = v3(ctl->T_ref[4], ctl->T_ref[5], ctl->T_ref[6]);
      const SE3q T_cur = se3_mul(model, T_ref);  // :92
      se3_store(T_cur, a.out_T + (size_t)b * 7);
      a.out_n_tracked[b] = ctl->n_meas_last / 16;  // :94
      for (int i = 0; i < 36; ++i) a.out_H[(size_t)b * 36 + i] = ctl->H_last[i];
      for (int l = 0; l < PLSVO_MAX_LEVELS; ++l) a.out_iters[(size_t)b * PLSVO_MAX_LEVELS + l] = ctl->iters_level[l];
      // status: bit 1 = solver stopped (NaN step); bits 2,3 = chi2 order could not be reproduced exactly (never
      // seen in practice; kept loud instead of silent)
      a.out_status[b] = (ctl->stop ? 2 : 0) | (ctl->chi2_flags << 2);
      a.out_patch_iters[b] = ctl->patch_iters;
      a.out_patch_levels[b] = ctl->patch_levels;
    }
  }
}

}  // namespace

namespace {
__global__ void weight_selftest_kernel(uint32_t n, uint32_t seed, unsigned long long* mismatch) {
  unsigned long long bad = 0;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    // half of the samples: random bit patterns in [0,256); other half: residual-like values k/2^m
    uint32_t h = (i ^ seed) * 2654435761u;
    h ^= h >> 15;
    h *= 2246822519u;
    h ^= h >> 13;
    float a;
    if (i & 1) {
      a = __uint_as_float(h % 0x43800000u);  // all floats in [0,256)
    } else {
      a = (float)(h & 0xffffff) * (1.0f / 65536.0f);  // multiples of 2^-16 below 256
    }
    const float fast = weight_rcp(a);
    const float ref = (float)(1.0 / (1.0 + (double)a));
    if (__float_as_uint(fast) != __float_as_uint(ref)) ++bad;
    // the packed form used by the kernel (both halves, either sign of the residual): exactly -w
    float n0, n1;
    upk2(neg_weight_rcp2(pk2(a, -a)), n0, n1);
    if (__float_as_uint(-n0) != __float_as_uint(ref) || __float_as_uint(-n1) != __float_as_uint(ref)) ++bad;
  }
  if (bad) atomicAdd(mismatch, bad);
}
}  // namespace

cudaError_t weight_selftest_launch(uint32_t n, uint32_t seed, unsigned long long* d_mismatch, cudaStream_t s) {
  weight_selftest_kernel<<<592, 256, 0, s>>>(n, seed, d_mismatch);
  return cudaGetLastError();
}

size_t align_smem_bytes(int n_pts, int n_segs, int max_patches, int max_seg_slots, int img_bytes, int threads) {
  return make_layout(n_pts, n_segs, max_patches, max_seg_slots, img_bytes, threads).total;
}

// Kernel variants: CTA size x resident CTAs per SM the register budget is compiled for.  Small CTAs with many
// resident pairs hide each pair's serial solve and barriers behind the other pairs and let a batch of ~7 pairs per
// SM run in a single wave; big CTAs cut the latency of a pair when the batch is small.
#define PLSVO_ALIGN_VARIANTS(X) X(64, 8) X(96, 7) X(96, 5) X(128, 5) X(128, 4) X(160, 3) X(192, 2) X(256, 2)

namespace {
template <int NT, int MINB>
cudaError_t prepare_t(size_t smem_bytes, int* ctas_per_sm) {
  cudaError_t e = cudaFuncSetAttribute(sparse_img_align_kernel<NT, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem_bytes);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(sparse_img_align_kernel<NT, MINB>, cudaFuncAttributePreferredSharedMemoryCarveout,
                           cudaSharedmemCarveoutMaxShared);
  if (e != cudaSuccess) return e;
  return cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctas_per_sm, sparse_img_align_kernel<NT, MINB>, NT, smem_bytes);
}
}  // namespace

cudaError_t align_kernel_prepare(int threads, int min_blocks, size_t smem_bytes, int* ctas_per_sm) {
#define X(NT, MB) \
  if (threads == NT && min_blocks == MB) return prepare_t<NT, MB>(smem_bytes, ctas_per_sm);
  PLSVO_ALIGN_VARIANTS(X)
#undef X
  return cudaErrorInvalidValue;
}

cudaError_t align_kernel_launch(const AlignArgs& a, int grid, int threads, int min_blocks, size_t smem_bytes,
                                cudaStream_t s) {
#define X(NT, MB)                                                            \
  if (threads == NT && min_blocks == MB) {                                   \
    sparse_img_align_kernel<NT, MB><<<grid, NT, smem_bytes, s>>>(a);         \
    return cudaGetLastError();                                               \
  }
  PLSVO_ALIGN_VARIANTS(X)
#undef X
  return cudaErrorInvalidValue;
}

}  // namespace plsvo
