// plsvo_abi.cu — the C ABI of include/plsvo_b200.h: context, host<->device staging, launches.
// Host-side only; the kernels are in align_kernel.cu and poseopt_kernel.cu.
#include <cuda_runtime.h>
#include <chrono>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <thread>
#include <vector>

#include "internal.h"

using namespace plsvo;

namespace {

thread_local std::string g_create_error;

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
};

struct plsvo_ctx_impl {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  cudaStream_t copy_stream = nullptr;  // second stream of the chunked host-buffer pipeline
  cudaStream_t rr_stream[4] = {nullptr, nullptr, nullptr, nullptr};  // extra copy streams: the arrays of a chunk go round-robin
  cudaEvent_t rr_ev[4] = {nullptr, nullptr, nullptr, nullptr};
  int rr_n = 0, rr_i = 0;  // rr_n > 0 only while the gated pipeline enqueues its copies
  cudaEvent_t chunk_ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t start_ev = nullptr;
  cudaEvent_t k_ev[2] = {nullptr, nullptr};  // around the kernel of the last pyramid / align2D / align1D call
  unsigned int* h_flags = nullptr;  // pinned arrival values of the gated pipeline
  char* h_out = nullptr;            // pinned staging of the alignment outputs (one D2H per download)
  size_t h_out_cap = 0, out_bytes = 0;
  size_t oo_T = 0, oo_H = 0, oo_ntr = 0, oo_iters = 0, oo_status = 0, oo_pi = 0, oo_pl = 0, oo_killed = 0;
  int h_flags_cap = 0;
  int num_sms = 0;
  int smem_optin = 0;
  std::string err;
  long long launches = 0;

  // ---- alignment state ----
  bool align_ready = false;
  AlignArgs aa;
  plsvo_camera cam;
  int a_max_seg_patches_l0 = 0;  // bound at level 0 (levels >= 0 never need more)
  std::vector<int> seg_patch_bound;  // per level: max over pairs of the number of segment samples
  std::vector<int> seg_slot_bound;   // per level: max over pairs of the lane slots of the segment groups
  std::vector<int> seg_maxN;         // per level: most samples of any one segment
  DevBuf d_ref_der, d_cur_der;       // pyramid levels derived on the device (vk::halfSample) instead of uploaded
  int der_src = -1, der_top = -1;    // derived levels are (der_src, der_top], built from uploaded level der_src
  bool lvl_uploaded[PLSVO_MAX_LEVELS] = {false};
  bool chain = false;              // PLSVO_ALIGN_FRAME_CHAIN: one stack of B+1 frames, cur(b) = frame b+1 = ref(b+1)
  DevBuf d_pt_depth, d_seg_sdepth, d_seg_edepth;
  DevBuf d_feat;                     // small batches: every feature array in one block (one host->device copy)
  char* h_po_out = nullptr;          // pinned staging of the pose-optimiser outputs (one D2H per download)
  size_t h_po_out_cap = 0, po_out_bytes = 0, po_zero_off = 0, po_zero_bytes = 0;
  DevBuf p_in;                       // packed inputs of a small pose-optimiser batch
  char* h_in = nullptr;              // pinned staging of the small-batch upload
  size_t h_in_cap = 0, img_total = 0;
  cudaEvent_t h_in_ev = nullptr;     // the staged copies of the previous small upload
  DevBuf d_ref_img, d_cur_img, d_T_ref, d_T_cur, d_pt_count, d_pt_px, d_pt_f, d_pt_pos, d_pt_valid, d_seg_count,
      d_seg_spx, d_seg_epx, d_seg_sf, d_seg_ef, d_seg_spos, d_seg_epos, d_seg_length, d_seg_valid;
  DevBuf d_out_T, d_out_ntr, d_out_H, d_out_killed, d_out_iters, d_out_status, d_out_pi, d_out_pl, d_counter,
      d_ws_cache, d_ws_xyz, d_ws_segpx, d_ws_rec, d_stage;
  DevBuf d_unit_done, d_unit_state;  // level units: per-pair progress words and the state carried between levels
  unsigned long long unit_epoch = 0;
  size_t level_off[PLSVO_MAX_LEVELS];

  // ---- pose-opt state ----
  bool po_ready = false;
  PoseOptArgs pa;
  DevBuf p_T, p_pt_count, p_pt_f, p_pt_pos, p_pt_level, p_pt_valid, p_seg_count, p_seg_line, p_seg_spos, p_seg_epos,
      p_seg_level, p_seg_valid;
  DevBuf y_img;  // pyramid levels
  DevBuf f_img, f_idx, f_lvl, f_border, f_ref, f_px, f_opx, f_oconv, f_dir, f_ohinv;  // align2D / align1D
  DevBuf m_ref_img, m_cur_img, m_T_ref, m_T_cur, m_ridx, m_cidx, m_px, m_f, m_lvl, m_edge, m_grad, m_pos, m_pxc, m_opx, m_osucc,
      m_olvl, m_oA;  // findMatchDirect
  DevBuf d_sa, d_sb, d_smu, d_szr, d_ssig, d_smu_e, d_szr_e, d_ssig_e, d_sout;  // depth-filter seeds
  DevBuf s_T, s_pb, s_pf, s_pof, s_pp, s_sb, s_sf, s_ssf, s_sef, s_sp, s_ep, s_out;  // structure optimisation
  DevBuf p_out_T, p_out_cov, p_out_scale, p_out_ei, p_out_ef, p_out_npt, p_out_nls, p_out_pto, p_out_sgo, p_out_iters,
      p_out_status;
};

#define CTX(c) reinterpret_cast<plsvo_ctx_impl*>(c)

int fail(plsvo_ctx_impl* c, int code, const char* what, cudaError_t e = cudaSuccess) {
  char buf[512];
  if (e != cudaSuccess)
    snprintf(buf, sizeof buf, "%s: %s (%s)", what, cudaGetErrorString(e), cudaGetErrorName(e));
  else
    snprintf(buf, sizeof buf, "%s", what);
  if (c)
    c->err = buf;
  else
    g_create_error = buf;
  return code;
}

#define CK(call)                                                        \
  do {                                                                  \
    cudaError_t e_ = (call);                                            \
    if (e_ != cudaSuccess) return fail(c, PLSVO_ERR_CUDA, #call, e_);   \
  } while (0)

// Records one of the two timing events around the kernel of a host-in/host-out entry point.
cudaError_t kernel_timer(plsvo_ctx_impl* c, int which, cudaStream_t s) {
  if (!c->k_ev[which]) {
    cudaError_t e = cudaEventCreate(&c->k_ev[which]);
    if (e != cudaSuccess) return e;
  }
  return cudaEventRecord(c->k_ev[which], s);
}

cudaError_t ensure(DevBuf& b, size_t bytes) {
  if (bytes <= b.cap && b.p) return cudaSuccess;
  if (b.p) cudaFree(b.p);
  b.p = nullptr;
  b.cap = 0;
  const size_t want = std::max<size_t>(bytes, 256);
  cudaError_t e = cudaMalloc(&b.p, want);
  if (e == cudaSuccess) b.cap = want;
  return e;
}

void release(DevBuf& b) {
  if (b.p) cudaFree(b.p);
  b.p = nullptr;
  b.cap = 0;
}

// upload a host array (or leave the device pointer NULL when the host pointer is NULL)
template <class T>
cudaError_t up(DevBuf& b, const T* host, size_t count, cudaStream_t s, const T** dev) {
  if (!host || count == 0) {
    *dev = nullptr;
    return cudaSuccess;
  }
  cudaError_t e = ensure(b, count * sizeof(T));
  if (e != cudaSuccess) return e;
  *dev = static_cast<const T*>(b.p);
  return cudaMemcpyAsync(b.p, host, count * sizeof(T), cudaMemcpyHostToDevice, s);
}

// LineFeat::setupSampling + per-level decimation on the host, to size the segment-sample slots
// (reference: src/feature.cpp:160-173, src/sparse_img_align.cpp:318-320)
int host_seg_samples(const double* spx, const double* epx, double length, int level) {
  const double d0 = fabs(epx[0] - spx[0]), d1 = fabs(epx[1] - spx[1]);
  const double tan_dir = std::min(d0, d1) / std::max(d0, d1);
  const double sin_dir = tan_dir / sqrt(1.0 + tan_dir * tan_dir);
  const double correction = 2.0 * sqrt(1.0 + sin_dir * sin_dir);
  double nd = length / (2.0 * 4 * correction);
  if (!(nd >= 1.0)) nd = 1.0;  // also catches NaN
  if (nd > 1e6) nd = 1e6;
  const unsigned long long n0 = (unsigned long long)nd;
  return (int)(1 + (n0 - 1) / (unsigned long long)(1 << level));
}

// The host-in/host-out entry points (plsvo_*_batch_run) promise that the caller's arrays are not read once they have
// returned — also when they return an error after copies have been queued (a level that can neither be found nor derived, a
// count out of range found by the sizing pass, ...).  Every such entry point passes its result through here: a non-OK
// result first drains every stream of the context (tests/test_host_pipeline_cpu.py counts pending host reads).
int settled(plsvo_ctx_impl* c, int rc) {
  if (rc == PLSVO_OK || !c) return rc;
  if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
  for (int k = 0; k < 4; ++k)
    if (c->rr_stream[k]) cudaStreamSynchronize(c->rr_stream[k]);
  cudaStreamSynchronize(c->stream);
  return rc;
}

}  // namespace

extern "C" {

const char* plsvo_version(void) { return "plsvo_b200 0.1.0 sm_100a"; }

int plsvo_ctx_create(int device, void* stream, plsvo_ctx** out) {
  if (!out) return PLSVO_ERR_INVALID;
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    return fail(nullptr, PLSVO_ERR_NO_DEVICE, "no CUDA device available (there is no CPU fallback)", e);
  if (device < 0 || device >= n) return fail(nullptr, PLSVO_ERR_INVALID, "device ordinal out of range");
  e = cudaSetDevice(device);
  if (e != cudaSuccess) return fail(nullptr, PLSVO_ERR_CUDA, "cudaSetDevice", e);
  plsvo_ctx_impl* c = new plsvo_ctx_impl();
  c->device = device;
  cudaDeviceGetAttribute(&c->num_sms, cudaDevAttrMultiProcessorCount, device);
  cudaDeviceGetAttribute(&c->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
  if (stream) {
    c->stream = static_cast<cudaStream_t>(stream);
  } else {
    e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
      delete c;
      return fail(nullptr, PLSVO_ERR_CUDA, "cudaStreamCreate", e);
    }
    c->own_stream = true;
  }
  memset(&c->aa, 0, sizeof c->aa);
  memset(&c->pa, 0, sizeof c->pa);
  *out = reinterpret_cast<plsvo_ctx*>(c);
  return PLSVO_OK;
}

void plsvo_ctx_destroy(plsvo_ctx* ctx) {
  if (!ctx) return;
  plsvo_ctx_impl* c = CTX(ctx);
  cudaSetDevice(c->device);
  // nothing may still be writing into the buffers freed below: the copy streams first, then the main stream
  if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
  for (int k = 0; k < 4; ++k)
    if (c->rr_stream[k]) cudaStreamSynchronize(c->rr_stream[k]);
  cudaStreamSynchronize(c->stream);
  DevBuf* bufs[] = {&c->d_ref_img,   &c->d_cur_img,  &c->d_T_ref,     &c->d_T_cur,      &c->d_pt_count,  &c->d_pt_px,
                    &c->d_pt_f,      &c->d_pt_pos,   &c->d_pt_valid,  &c->d_seg_count,  &c->d_seg_spx,   &c->d_seg_epx,
                    &c->d_seg_sf,    &c->d_seg_ef,   &c->d_seg_spos,  &c->d_seg_epos,   &c->d_seg_length, &c->d_seg_valid,
                    &c->d_out_T,     &c->d_out_ntr,  &c->d_out_H,     &c->d_out_killed, &c->d_out_iters, &c->d_out_status,
                    &c->d_out_pi,    &c->d_out_pl,   &c->d_counter,   &c->d_ws_cache,   &c->d_ws_xyz,    &c->d_ref_der,   &c->d_cur_der,   &c->d_pt_depth,  &c->d_seg_sdepth, &c->d_seg_edepth, &c->d_feat, &c->d_ws_segpx,  &c->d_ws_rec,    &c->d_stage,     &c->d_unit_done, &c->d_unit_state, &c->y_img,       &c->f_img,       &c->f_idx,       &c->f_lvl,      &c->f_border,
                    &c->f_ref,       &c->f_px,        &c->f_opx,       &c->f_oconv,     &c->f_dir,       &c->f_ohinv,     &c->m_ref_img,   &c->m_cur_img,   &c->m_T_ref,     &c->m_T_cur,
                    &c->m_ridx,      &c->m_cidx,     &c->m_px,        &c->m_f,          &c->m_lvl,       &c->m_edge,
                    &c->m_grad,      &c->m_pos,      &c->m_pxc,       &c->m_opx,        &c->m_osucc,     &c->m_olvl,      &c->m_oA,        &c->s_T,         &c->s_pb,        &c->s_pf,        &c->s_pof,
                    &c->s_pp,        &c->s_sb,       &c->s_sf,        &c->s_ssf,        &c->s_sef,       &c->s_sp,
                    &c->s_ep,        &c->s_out,      &c->d_sa,        &c->d_sb,         &c->d_smu,       &c->d_szr,
                    &c->d_ssig,      &c->d_smu_e,    &c->d_szr_e,     &c->d_ssig_e,     &c->d_sout,      &c->p_T,
                    &c->p_pt_count,  &c->p_pt_f,     &c->p_pt_pos,    &c->p_pt_level,   &c->p_pt_valid,  &c->p_seg_count,
                    &c->p_seg_line,  &c->p_seg_spos, &c->p_seg_epos,  &c->p_seg_level,  &c->p_seg_valid, &c->p_out_T,
                    &c->p_out_cov,   &c->p_out_scale, &c->p_out_ei,   &c->p_out_ef,     &c->p_out_npt,   &c->p_out_nls,
                    &c->p_out_pto,   &c->p_out_sgo,  &c->p_out_iters, &c->p_out_status};
  for (DevBuf* b : bufs) release(*b);
  if (c->h_flags) cudaFreeHost(c->h_flags);
  if (c->h_out) cudaFreeHost(c->h_out);
  if (c->h_in) cudaFreeHost(c->h_in);
  if (c->h_po_out) cudaFreeHost(c->h_po_out);
  release(c->p_in);
  if (c->h_in_ev) cudaEventDestroy(c->h_in_ev);
  for (int k = 0; k < 4; ++k) {
    if (c->rr_stream[k]) cudaStreamDestroy(c->rr_stream[k]);
    if (c->rr_ev[k]) cudaEventDestroy(c->rr_ev[k]);
  }
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  for (int k = 0; k < 8; ++k)
    if (c->chunk_ev[k]) cudaEventDestroy(c->chunk_ev[k]);
  if (c->start_ev) cudaEventDestroy(c->start_ev);
  for (auto& e : c->k_ev)
    if (e) cudaEventDestroy(e);
  if (c->own_stream) cudaStreamDestroy(c->stream);
  delete c;
}

const char* plsvo_last_error(const plsvo_ctx* ctx) {
  if (!ctx) return g_create_error.c_str();
  return reinterpret_cast<const plsvo_ctx_impl*>(ctx)->err.c_str();
}

void* plsvo_ctx_stream(plsvo_ctx* ctx) { return ctx ? (void*)CTX(ctx)->stream : nullptr; }

int plsvo_sync(plsvo_ctx* ctx) {
  if (!ctx) return PLSVO_ERR_INVALID;
  plsvo_ctx_impl* c = CTX(ctx);
  CK(cudaStreamSynchronize(c->stream));
  return PLSVO_OK;
}

int plsvo_host_alloc(void** ptr, size_t bytes) {
  if (!ptr) return PLSVO_ERR_INVALID;
  cudaError_t e = cudaHostAlloc(ptr, bytes, cudaHostAllocDefault);
  if (e != cudaSuccess) {
    *ptr = nullptr;
    return fail(nullptr, e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver ? PLSVO_ERR_NO_DEVICE : PLSVO_ERR_CUDA,
                "cudaHostAlloc", e);
  }
  return PLSVO_OK;
}
int plsvo_host_free(void* ptr) {
  if (!ptr) return PLSVO_OK;
  return cudaFreeHost(ptr) == cudaSuccess ? PLSVO_OK : PLSVO_ERR_CUDA;
}

int plsvo_last_kernel_ms(plsvo_ctx* ctx, float* ms) {
  if (!ctx || !ms) return PLSVO_ERR_INVALID;
  plsvo_ctx_impl* c = CTX(ctx);
  if (!c->k_ev[0] || !c->k_ev[1]) return fail(c, PLSVO_ERR_STATE, "no timed kernel has run on this context");
  CK(cudaEventSynchronize(c->k_ev[1]));
  CK(cudaEventElapsedTime(ms, c->k_ev[0], c->k_ev[1]));
  return PLSVO_OK;
}

int64_t plsvo_launch_count(const plsvo_ctx* ctx) {
  return ctx ? reinterpret_cast<const plsvo_ctx_impl*>(ctx)->launches : 0;
}

int plsvo_selftest_weight(plsvo_ctx* ctx, uint32_t n, uint32_t seed, uint64_t* mismatches) {
  if (!ctx || !mismatches) return PLSVO_ERR_INVALID;
  plsvo_ctx_impl* c = CTX(ctx);
  CK(cudaSetDevice(c->device));
  CK(ensure(c->d_counter, 256));
  unsigned long long* d = reinterpret_cast<unsigned long long*>(static_cast<char*>(c->d_counter.p) + 64);
  CK(cudaMemsetAsync(d, 0, sizeof(unsigned long long), c->stream));
  CK(weight_selftest_launch(n, seed, d, c->stream));
  c->launches += 1;
  unsigned long long h = 0;
  CK(cudaMemcpyAsync(&h, d, sizeof h, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  *mismatches = h;
  return PLSVO_OK;
}

// ------------------------------------------------------------------------------------------------
// alignment
// ------------------------------------------------------------------------------------------------
}  // extern "C" (helpers below use templates)

namespace {

// copy items [b0,b1) of a per-pair host array to its device buffer (device pointer NULL when the host one is)
template <class T>
cudaError_t up_range(DevBuf& buf, const T* host, size_t per_item, size_t B, size_t b0, size_t b1, cudaStream_t s,
                     const T** dev, bool prepare) {
  if (!host || per_item == 0) {
    *dev = nullptr;
    return cudaSuccess;
  }
  if (prepare) {
    cudaError_t e = ensure(buf, B * per_item * sizeof(T));
    if (e != cudaSuccess) return e;
  }
  *dev = static_cast<const T*>(buf.p);
  return cudaMemcpyAsync(static_cast<T*>(buf.p) + b0 * per_item, host + b0 * per_item, (b1 - b0) * per_item * sizeof(T),
                         cudaMemcpyHostToDevice, s);
}

// Host arrays -> device layout for pairs [b0,b1).  prepare = validate, size the buffers for the whole batch
// and lay out the pyramid levels; later chunks of the same batch only copy.
// Stream for the next host->device array copy: the caller's stream, or — while the gated pipeline is enqueuing a chunk —
// one of the extra copy streams in turn, so that the per-copy start-up latency of one array overlaps the transfer of another.
static inline cudaStream_t pick_copy_stream(plsvo_ctx_impl* c, cudaStream_t s) {
  if (c->rr_n <= 0 || s != c->copy_stream) return s;
  return c->rr_stream[c->rr_i++ % c->rr_n];
}

int align_upload_impl(plsvo_ctx_impl* c, const plsvo_align_batch* h, size_t b0, size_t b1, cudaStream_t s, int mode,
                      int what = 3, int size_level = -1) {
  // mode 0: copy [b0,b1) only; 1: validate + lay out + copy + host-side sizing; 2: validate + lay out + copy;
  // 3: host-side sizing only.  what: bit 0 = the image levels, bit 1 = the feature arrays (the streamed host path sends
  // every feature array of the batch first and then the images chunk by chunk).  size_level >= 0: the sizing is wanted for
  // that pyramid level only and may be a cheap upper bound (it sits on the launch path of the streamed host call).
  AlignArgs& a = c->aa;
  const size_t B = (size_t)h->batch;
  const bool prepare = (mode == 1 || mode == 2);
  if (mode != 3) {
  if (prepare) {
    c->align_ready = false;
    if (h->batch <= 0 || h->n_pts < 0 || h->n_segs < 0 || h->n_segs > 32767)
      return fail(c, PLSVO_ERR_INVALID, "batch/n_pts/n_segs out of range");
    if (!h->T_ref_w || !h->T_cur_w) return fail(c, PLSVO_ERR_INVALID, "T_ref_w/T_cur_w missing");
    if (h->n_pts > 0 && (!h->pt_px || (!h->pt_pos && !h->pt_depth)))
      return fail(c, PLSVO_ERR_INVALID, "point arrays missing");
    if (h->n_segs > 0 && (!h->seg_spx || !h->seg_epx || (!h->seg_spos && !h->seg_sdepth) ||
                          (!h->seg_epos && !h->seg_edepth) || !h->seg_length))
      return fail(c, PLSVO_ERR_INVALID, "segment arrays missing");
    if (h->cam.width <= 0 || h->cam.height <= 0) return fail(c, PLSVO_ERR_INVALID, "camera size");
    if (h->flags & ~PLSVO_ALIGN_FRAME_CHAIN) return fail(c, PLSVO_ERR_INVALID, "unknown bits in plsvo_align_batch.flags");
    CK(cudaSetDevice(c->device));
    // frame chain: ref_img[l] is one stack of B+1 frames and the current image of pair b is frame b+1 — the kernel's
    // `cur_img[l] + b*stride` then simply starts one frame further into the same stack
    c->chain = (h->flags & PLSVO_ALIGN_FRAME_CHAIN) != 0;
    const size_t n_frames = B + (c->chain ? 1 : 0);
    a.B = h->batch, a.n_pts = h->n_pts, a.n_segs = h->n_segs;
    a.width = h->cam.width, a.height = h->cam.height;
    a.fx = h->cam.fx, a.fy = h->cam.fy, a.cx = h->cam.cx, a.cy = h->cam.cy;
    c->cam = h->cam;
    // images: every provided level is packed as [B][rows][pitch16]
    size_t total = 0;
    for (int l = 0; l < PLSVO_MAX_LEVELS; ++l) {
      a.ref_img[l] = a.cur_img[l] = nullptr;
      a.pitch[l] = 0, a.stride[l] = 0;
      c->level_off[l] = 0;
      c->lvl_uploaded[l] = false;
      if (!h->ref_img[l] || (!c->chain && !h->cur_img[l])) continue;
      c->lvl_uploaded[l] = true;
      const int cols = h->cam.width >> l, rows = h->cam.height >> l;
      if (cols <= 0 || rows <= 0) return fail(c, PLSVO_ERR_INVALID, "pyramid level smaller than one pixel");
      if (h->img_pitch[l] < (size_t)cols) return fail(c, PLSVO_ERR_INVALID, "img_pitch smaller than the level width");
      // device pitch: the host layout is kept when rows are word aligned and images 16-byte aligned
      // (what the aligned-word loads and the bulk copy need) — then a level moves with one linear copy;
      // otherwise rows are padded to 16 bytes and repacked on the device.
      uint32_t pitch = (uint32_t)((cols + 15) / 16 * 16);
      const bool uniform = h->img_stride[l] == (size_t)rows * h->img_pitch[l];
      if (uniform && h->img_pitch[l] % 4 == 0 && h->img_stride[l] % 16 == 0 && h->img_pitch[l] < (1u << 20))
        pitch = (uint32_t)h->img_pitch[l];
      a.pitch[l] = pitch;
      a.stride[l] = (size_t)rows * pitch;
      total = (total + 255) / 256 * 256;
      c->level_off[l] = total;
      total += a.stride[l] * n_frames;
    }
    CK(ensure(c->d_ref_img, total + 256));
    if (!c->chain) CK(ensure(c->d_cur_img, total + 256));
    c->img_total = total;
    c->der_src = c->der_top = -1;
    size_t stage = 0;
    for (int l = 0; l < PLSVO_MAX_LEVELS; ++l)
      if (a.pitch[l] && h->img_pitch[l] != a.pitch[l]) stage = std::max(stage, 2 * h->img_stride[l] * n_frames);
    if (stage) CK(ensure(c->d_stage, stage));
  }
  // ---- small batches (the reference's own call is B = 1, frame_handler_mono.cpp:272): every input is packed into one
  // pinned staging block and moves with three copies (reference images, current images, all feature arrays) instead of
  // ~20 separate copies from pageable memory, each of which costs more than the kernel of a single pair ----
  {
    const size_t np_ = (size_t)h->n_pts, ns_ = (size_t)h->n_segs;
    struct Item {
      const void* host;
      size_t bytes;
      const void** dev;
    };
    const Item items[] = {
        {h->T_ref_w, B * 7 * 8, (const void**)&a.T_ref_w},
        {h->T_cur_w, B * 7 * 8, (const void**)&a.T_cur_w},
        {h->pt_count, B * 4, (const void**)&a.pt_count},
        {h->pt_px, B * np_ * 16, (const void**)&a.pt_px},
        {h->pt_f, B * np_ * 24, (const void**)&a.pt_f},
        {h->pt_depth ? nullptr : h->pt_pos, B * np_ * 24, (const void**)&a.pt_pos},
        {h->pt_depth, B * np_ * 8, (const void**)&a.pt_depth},
        {h->pt_valid, B * np_, (const void**)&a.pt_valid},
        {h->seg_count, B * 4, (const void**)&a.seg_count},
        {h->seg_spx, B * ns_ * 16, (const void**)&a.seg_spx},
        {h->seg_epx, B * ns_ * 16, (const void**)&a.seg_epx},
        {h->seg_sf, B * ns_ * 24, (const void**)&a.seg_sf},
        {h->seg_ef, B * ns_ * 24, (const void**)&a.seg_ef},
        {h->seg_sdepth ? nullptr : h->seg_spos, B * ns_ * 24, (const void**)&a.seg_spos},
        {h->seg_edepth ? nullptr : h->seg_epos, B * ns_ * 24, (const void**)&a.seg_epos},
        {h->seg_sdepth, B * ns_ * 8, (const void**)&a.seg_sdepth},
        {h->seg_edepth, B * ns_ * 8, (const void**)&a.seg_edepth},
        {h->seg_length, B * ns_ * 8, (const void**)&a.seg_length},
        {h->seg_valid, B * ns_, (const void**)&a.seg_valid},
    };
    size_t feat_total = 0;
    for (const Item& it : items)
      if (it.host && it.bytes) feat_total += (it.bytes + 255) / 256 * 256;
    bool small = prepare && what == 3 && b0 == 0 && b1 == B && c->rr_n == 0 && s == c->stream && !getenv("PLSVO_NO_SMALL_UPLOAD") &&
                 2 * c->img_total + feat_total <= (size_t)4 << 20;
    for (int l = 0; l < PLSVO_MAX_LEVELS && small; ++l) {
      if (!c->lvl_uploaded[l]) continue;
      const int rows = h->cam.height >> l;
      if (!(h->img_stride[l] == (size_t)rows * h->img_pitch[l] && h->img_pitch[l] == a.pitch[l])) small = false;  // needs the repack path
    }
    if (small) {
      const size_t need = 2 * c->img_total + feat_total + 256;
      if (c->h_in_cap < need) {
        if (c->h_in_ev) CK(cudaEventSynchronize(c->h_in_ev));  // a copy out of the old block may still be queued
        if (c->h_in) cudaFreeHost(c->h_in);
        c->h_in = nullptr, c->h_in_cap = 0;
        CK(cudaHostAlloc((void**)&c->h_in, need, cudaHostAllocDefault));
        c->h_in_cap = need;
      }
      if (!c->h_in_ev) CK(cudaEventCreateWithFlags(&c->h_in_ev, cudaEventDisableTiming));
      else CK(cudaEventSynchronize(c->h_in_ev));  // the previous upload's copies have left the staging block
      CK(ensure(c->d_feat, feat_total + 256));
      char* hr = c->h_in;
      char* hc = c->h_in + c->img_total;
      char* hf = c->h_in + 2 * c->img_total;
      for (int l = 0; l < PLSVO_MAX_LEVELS; ++l) {
        if (!c->lvl_uploaded[l]) continue;
        memcpy(hr + c->level_off[l], h->ref_img[l], a.stride[l] * (B + (c->chain ? 1 : 0)));
        a.ref_img[l] = static_cast<uint8_t*>(c->d_ref_img.p) + c->level_off[l];
        if (c->chain) {
          a.cur_img[l] = a.ref_img[l] + a.stride[l];
          continue;
        }
        memcpy(hc + c->level_off[l], h->cur_img[l], a.stride[l] * B);
        a.cur_img[l] = static_cast<uint8_t*>(c->d_cur_img.p) + c->level_off[l];
      }
      size_t off = 0;
      for (const Item& it : items) {
        if (!it.host || !it.bytes) {
          *it.dev = nullptr;
          continue;
        }
        memcpy(hf + off, it.host, it.bytes);
        *it.dev = static_cast<char*>(c->d_feat.p) + off;
        off += (it.bytes + 255) / 256 * 256;
      }
      if (c->img_total) {
        CK(cudaMemcpyAsync(c->d_ref_img.p, hr, c->img_total, cudaMemcpyHostToDevice, s));
        if (!c->chain) CK(cudaMemcpyAsync(c->d_cur_img.p, hc, c->img_total, cudaMemcpyHostToDevice, s));
      }
      if (feat_total) CK(cudaMemcpyAsync(c->d_feat.p, hf, feat_total, cudaMemcpyHostToDevice, s));
      CK(cudaEventRecord(c->h_in_ev, s));
      goto copies_done;
    }
  }
  {
  const size_t nb = b1 - b0;
  for (int l = 0; l < PLSVO_MAX_LEVELS; ++l) {
    if (!c->lvl_uploaded[l]) continue;
    const int cols = h->cam.width >> l, rows = h->cam.height >> l;
    uint8_t* dr = static_cast<uint8_t*>(c->d_ref_img.p) + c->level_off[l];
    a.ref_img[l] = dr;
    const bool uniform = h->img_stride[l] == (size_t)rows * h->img_pitch[l];
    if (c->chain) {
      // pairs [b0,b1) read frames [b0, b1]: frame b0 came with the previous range (or is frame 0 of the first one)
      a.cur_img[l] = dr + a.stride[l];
      if (!(what & 1) || nb == 0) continue;
      const size_t f0 = b0 ? b0 + 1 : 0, nf = b1 + 1 - f0;
      const uint8_t* hf = h->ref_img[l] + f0 * h->img_stride[l];
      uint8_t* df = dr + f0 * a.stride[l];
      if (uniform && h->img_pitch[l] == a.pitch[l]) {
        CK(cudaMemcpyAsync(df, hf, a.stride[l] * nf, cudaMemcpyHostToDevice, pick_copy_stream(c, s)));
      } else if (uniform) {
        uint8_t* st = static_cast<uint8_t*>(c->d_stage.p) + h->img_stride[l] * f0;
        CK(cudaMemcpyAsync(st, hf, h->img_stride[l] * nf, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpy2DAsync(df, a.pitch[l], st, h->img_pitch[l], cols, (size_t)rows * nf, cudaMemcpyDeviceToDevice, s));
      } else {
        for (size_t k = 0; k < nf; ++k)
          CK(cudaMemcpy2DAsync(df + k * a.stride[l], a.pitch[l], hf + k * h->img_stride[l], h->img_pitch[l], cols, rows,
                               cudaMemcpyHostToDevice, s));
      }
      continue;
    }
    uint8_t* dc = static_cast<uint8_t*>(c->d_cur_img.p) + c->level_off[l];
    a.cur_img[l] = dc;
    const uint8_t* hr = h->ref_img[l] + b0 * h->img_stride[l];
    const uint8_t* hc = h->cur_img[l] + b0 * h->img_stride[l];
    dr += b0 * a.stride[l];
    dc += b0 * a.stride[l];
    if (!(what & 1) || nb == 0) continue;
    if (uniform && h->img_pitch[l] == a.pitch[l]) {
      // host stack already has the device layout: one linear copy per frame set
      CK(cudaMemcpyAsync(dr, hr, a.stride[l] * nb, cudaMemcpyHostToDevice, pick_copy_stream(c, s)));
      CK(cudaMemcpyAsync(dc, hc, a.stride[l] * nb, cudaMemcpyHostToDevice, pick_copy_stream(c, s)));
    } else if (uniform) {
      // uniformly pitched stack with a different pitch: linear H2D into staging (PCIe-friendly), then a
      // device-side 2D repack into the 16-byte-pitched layout (row-granular DMA over PCIe is slow)
      const size_t off = 2 * h->img_stride[l] * b0, bytes = h->img_stride[l] * nb;
      uint8_t* st = static_cast<uint8_t*>(c->d_stage.p) + off;
      CK(cudaMemcpyAsync(st, hr, bytes, cudaMemcpyHostToDevice, s));
      CK(cudaMemcpyAsync(st + bytes, hc, bytes, cudaMemcpyHostToDevice, s));
      CK(cudaMemcpy2DAsync(dr, a.pitch[l], st, h->img_pitch[l], cols, (size_t)rows * nb, cudaMemcpyDeviceToDevice, s));
      CK(cudaMemcpy2DAsync(dc, a.pitch[l], st + bytes, h->img_pitch[l], cols, (size_t)rows * nb, cudaMemcpyDeviceToDevice, s));
    } else {
      for (size_t b = 0; b < nb; ++b) {
        CK(cudaMemcpy2DAsync(dr + b * a.stride[l], a.pitch[l], hr + b * h->img_stride[l], h->img_pitch[l], cols, rows,
                             cudaMemcpyHostToDevice, s));
        CK(cudaMemcpy2DAsync(dc + b * a.stride[l], a.pitch[l], hc + b * h->img_stride[l], h->img_pitch[l], cols, rows,
                             cudaMemcpyHostToDevice, s));
      }
    }
  }
  const size_t np = (size_t)h->n_pts, ns = (size_t)h->n_segs;
  if (what & 2) {
  CK(up_range(c->d_T_ref, h->T_ref_w, 7, B, b0, b1, pick_copy_stream(c, s), &a.T_ref_w, prepare));
  CK(up_range(c->d_T_cur, h->T_cur_w, 7, B, b0, b1, pick_copy_stream(c, s), &a.T_cur_w, prepare));
  CK(up_range(c->d_pt_count, h->pt_count, 1, B, b0, b1, pick_copy_stream(c, s), &a.pt_count, prepare));
  CK(up_range(c->d_pt_px, h->pt_px, np * 2, B, b0, b1, pick_copy_stream(c, s), &a.pt_px, prepare));
  CK(up_range(c->d_pt_f, h->pt_f, np * 3, B, b0, b1, pick_copy_stream(c, s), &a.pt_f, prepare));
  CK(up_range(c->d_pt_pos, h->pt_depth ? nullptr : h->pt_pos, np * 3, B, b0, b1, pick_copy_stream(c, s), &a.pt_pos, prepare));
  CK(up_range(c->d_pt_depth, h->pt_depth, np, B, b0, b1, pick_copy_stream(c, s), &a.pt_depth, prepare));
  CK(up_range(c->d_pt_valid, h->pt_valid, np, B, b0, b1, pick_copy_stream(c, s), &a.pt_valid, prepare));
  CK(up_range(c->d_seg_count, h->seg_count, 1, B, b0, b1, pick_copy_stream(c, s), &a.seg_count, prepare));
  CK(up_range(c->d_seg_spx, h->seg_spx, ns * 2, B, b0, b1, pick_copy_stream(c, s), &a.seg_spx, prepare));
  CK(up_range(c->d_seg_epx, h->seg_epx, ns * 2, B, b0, b1, pick_copy_stream(c, s), &a.seg_epx, prepare));
  CK(up_range(c->d_seg_sf, h->seg_sf, ns * 3, B, b0, b1, pick_copy_stream(c, s), &a.seg_sf, prepare));
  CK(up_range(c->d_seg_ef, h->seg_ef, ns * 3, B, b0, b1, pick_copy_stream(c, s), &a.seg_ef, prepare));
  CK(up_range(c->d_seg_spos, h->seg_sdepth ? nullptr : h->seg_spos, ns * 3, B, b0, b1, pick_copy_stream(c, s), &a.seg_spos, prepare));
  CK(up_range(c->d_seg_epos, h->seg_edepth ? nullptr : h->seg_epos, ns * 3, B, b0, b1, pick_copy_stream(c, s), &a.seg_epos, prepare));
  CK(up_range(c->d_seg_sdepth, h->seg_sdepth, ns, B, b0, b1, pick_copy_stream(c, s), &a.seg_sdepth, prepare));
  CK(up_range(c->d_seg_edepth, h->seg_edepth, ns, B, b0, b1, pick_copy_stream(c, s), &a.seg_edepth, prepare));
  CK(up_range(c->d_seg_length, h->seg_length, ns, B, b0, b1, pick_copy_stream(c, s), &a.seg_length, prepare));
  CK(up_range(c->d_seg_valid, h->seg_valid, ns, B, b0, b1, pick_copy_stream(c, s), &a.seg_valid, prepare));
  }
  }
copies_done:;
  }  // mode != 3
  if (mode == 0 || mode == 2) return PLSVO_OK;

  // per-pair feature counts index shared memory and the feature arrays in the kernels: reject anything outside
  // [0, n_pts] / [0, n_segs] here (every other index array of the ABI is range-checked on the host as well)
  for (size_t b = 0; b < B; ++b) {
    if (h->pt_count && (h->pt_count[b] < 0 || h->pt_count[b] > h->n_pts))
      return fail(c, PLSVO_ERR_INVALID, "pt_count[b] outside [0, n_pts]");
    if (h->seg_count && (h->seg_count[b] < 0 || h->seg_count[b] > h->n_segs))
      return fail(c, PLSVO_ERR_INVALID, "seg_count[b] outside [0, n_segs]");
  }
  // per-level bounds on the segment samples of a pair: sample slots, lane slots of the segment groups (a segment
  // with N samples owns 2^k >= min(N,32) lanes) and the longest segment (host arrays are still valid here)
  c->seg_patch_bound.assign(PLSVO_MAX_LEVELS, 0);
  c->seg_slot_bound.assign(PLSVO_MAX_LEVELS, 0);
  c->seg_maxN.assign(PLSVO_MAX_LEVELS, 0);
  if (h->n_segs > 0) {
    // a few host threads: the sizing sits between the enqueued copies and the kernel launch of the host-buffer path
    struct Bounds {
      int patches[PLSVO_MAX_LEVELS], slots[PLSVO_MAX_LEVELS], maxN[PLSVO_MAX_LEVELS];
    };
    const bool fast = size_level >= 0 && size_level < PLSVO_MAX_LEVELS;
    const int nt = fast ? (int)std::max<size_t>(1, std::min<size_t>(4, B * (size_t)h->n_segs / 262144))
                        : (int)std::max<size_t>(1, std::min<size_t>(8, B * (size_t)h->n_segs / 8192));
    std::vector<Bounds> part(nt);
    auto work = [&](int t) {
      Bounds bd;
      memset(&bd, 0, sizeof bd);
      if (fast) {
        // Upper bound without the square roots and divisions of setupSampling: correction = 2 sqrt(1 + sin^2) >= 2, so the
        // sample count length / (2 * 4 * correction) is at most length / 16 (NaN or tiny lengths give 1, as on the device).
        const int l = size_level;
        int best_sum = 0, best_slots = 0, best_N = 0;
        for (size_t b = B * t / nt; b < B * (t + 1) / nt; ++b) {
          const int nsb = h->seg_count ? h->seg_count[b] : h->n_segs;
          const double* len = h->seg_length + b * (size_t)h->n_segs;
          int sum = 0, slots = 0;
          for (int j = 0; j < nsb; ++j) {
            double nd = len[j] * 0.0625;
            nd = nd >= 1.0 ? nd : 1.0;  // also catches NaN
            nd = nd > 1e6 ? 1e6 : nd;
            const int N = 1 + (((int)nd - 1) >> l);
            const int g = 2 * N - 1;  // the group of a segment has 2^k >= min(N, 32) lanes: at most min(2N - 1, 32)
            sum += N, slots += g < 32 ? g : 32;
            best_N = N > best_N ? N : best_N;
          }
          best_sum = std::max(best_sum, sum), best_slots = std::max(best_slots, slots);
        }
        bd.patches[l] = best_sum, bd.slots[l] = best_slots, bd.maxN[l] = best_N;
        part[t] = bd;
        return;
      }
      for (size_t b = B * t / nt; b < B * (t + 1) / nt; ++b) {
        const int nsb = h->seg_count ? h->seg_count[b] : h->n_segs;
        int sum[PLSVO_MAX_LEVELS] = {0}, slots[PLSVO_MAX_LEVELS] = {0};
        for (int j = 0; j < nsb; ++j) {
          const size_t k = b * h->n_segs + j;
          const int n0 = host_seg_samples(h->seg_spx + 2 * k, h->seg_epx + 2 * k, h->seg_length[k], 0);
          for (int l = 0; l < PLSVO_MAX_LEVELS; ++l) {
            const int N = 1 + ((n0 - 1) >> l);
            int g = 1;
            while (g < N && g < 32) g <<= 1;
            sum[l] += N;
            slots[l] += g;
            bd.maxN[l] = std::max(bd.maxN[l], N);
          }
        }
        for (int l = 0; l < PLSVO_MAX_LEVELS; ++l) {
          bd.patches[l] = std::max(bd.patches[l], sum[l]);
          bd.slots[l] = std::max(bd.slots[l], slots[l]);
        }
      }
      part[t] = bd;
    };
    if (nt == 1) {
      work(0);
    } else {
      std::vector<std::thread> pool;
      for (int t = 1; t < nt; ++t) pool.emplace_back(work, t);
      work(0);
      for (auto& th : pool) th.join();
    }
    for (const Bounds& bd : part)
      for (int l = 0; l < PLSVO_MAX_LEVELS; ++l) {
        c->seg_patch_bound[l] = std::max(c->seg_patch_bound[l], bd.patches[l]);
        c->seg_slot_bound[l] = std::max(c->seg_slot_bound[l], bd.slots[l]);
        c->seg_maxN[l] = std::max(c->seg_maxN[l], bd.maxN[l]);
      }
  }
  // all outputs live in one device block so that the download is a single D2H into pinned staging
  {
    const size_t nsg = (size_t)std::max(1, h->n_segs);
    size_t o = 0;
    auto take = [&](size_t bytes) { const size_t at = o; o = (o + bytes + 255) / 256 * 256; return at; };
    c->oo_T = take(B * 7 * sizeof(double));
    c->oo_H = take(B * 36 * sizeof(double));
    c->oo_ntr = take(B * sizeof(long long));
    c->oo_iters = take(B * PLSVO_MAX_LEVELS * sizeof(int32_t));
    c->oo_status = take(B * sizeof(int32_t));
    c->oo_pi = take(B * sizeof(uint32_t));
    c->oo_pl = take(B * sizeof(uint32_t));
    c->oo_killed = take(B * nsg);
    c->out_bytes = o;
    CK(ensure(c->d_out_T, o));
    if (c->h_out_cap < o) {
      if (c->h_out) cudaFreeHost(c->h_out);
      c->h_out = nullptr, c->h_out_cap = 0;
      CK(cudaHostAlloc((void**)&c->h_out, o, cudaHostAllocDefault));
      c->h_out_cap = o;
    }
    char* base = static_cast<char*>(c->d_out_T.p);
    a.out_T = reinterpret_cast<double*>(base + c->oo_T);
    a.out_H = reinterpret_cast<double*>(base + c->oo_H);
    a.out_n_tracked = reinterpret_cast<long long*>(base + c->oo_ntr);
    a.out_iters = reinterpret_cast<int32_t*>(base + c->oo_iters);
    a.out_status = reinterpret_cast<int32_t*>(base + c->oo_status);
    a.out_patch_iters = reinterpret_cast<uint32_t*>(base + c->oo_pi);
    a.out_patch_levels = reinterpret_cast<uint32_t*>(base + c->oo_pl);
    a.out_seg_killed = reinterpret_cast<uint8_t*>(base + c->oo_killed);
  }
  CK(ensure(c->d_counter, 256));
  a.work_counter = static_cast<unsigned int*>(c->d_counter.p);
  c->align_ready = true;
  return PLSVO_OK;
}

// Pyramid levels that were not uploaded are derived on the device from the highest uploaded level below them by
// repeated vk::halfSample (pyramid_kernel.cu; bit-identical to frame_utils::createImgPyramid), for pairs [b0,b1).
// prepare: size the buffers and describe the derived levels in AlignArgs (once per batch).
int align_derive_levels(plsvo_ctx_impl* c, int min_level, int max_level, size_t b0, size_t b1, cudaStream_t s, bool prepare,
                        bool in_kernel = false) {
  AlignArgs& a = c->aa;
  a.derive_from = -1;
  int first_missing = -1;
  for (int l = min_level; l <= max_level; ++l)
    if (!c->lvl_uploaded[l]) {
      first_missing = l;
      break;
    }
  if (first_missing < 0) return PLSVO_OK;
  int src = -1;
  for (int l = first_missing - 1; l >= 0; --l)
    if (c->lvl_uploaded[l]) {
      src = l;
      break;
    }
  if (src < 0) return fail(c, PLSVO_ERR_INVALID, "a pyramid level in [min_level,max_level] was not uploaded and no lower level is there to derive it from");
  for (int l = first_missing; l <= max_level; ++l)
    if (c->lvl_uploaded[l]) return fail(c, PLSVO_ERR_INVALID, "derived pyramid levels must be contiguous above the uploaded ones");
  // the pyramid kernel reads 16-byte rows; a source level whose host layout was kept with a pitch that is only word aligned
  // (e.g. 188-byte rows: level 2 of a 752-pixel-wide camera) is halfSampled by the alignment kernel itself, pair by pair,
  // byte by byte — the same code the arrival-gated stream uses
  if (a.pitch[src] % 16 != 0 || a.stride[src] % 16 != 0) in_kernel = true;
  const size_t B = (size_t)a.B;
  if (prepare || c->der_src != src || c->der_top < max_level) {
    size_t total = 0, off[PLSVO_MAX_LEVELS] = {0};
    for (int l = src + 1; l <= max_level; ++l) {
      const int cols = a.width >> l, rows = a.height >> l;
      if (cols <= 0 || rows <= 0) return fail(c, PLSVO_ERR_INVALID, "pyramid level smaller than one pixel");
      a.pitch[l] = (uint32_t)((cols + 15) / 16 * 16);
      a.stride[l] = (size_t)rows * a.pitch[l];
      off[l] = total;
      total += (a.stride[l] * (B + (c->chain ? 1 : 0)) + 255) / 256 * 256;
    }
    CK(ensure(c->d_ref_der, total + 256));
    if (!c->chain) CK(ensure(c->d_cur_der, total + 256));
    for (int l = src + 1; l <= max_level; ++l) {
      a.ref_img[l] = static_cast<uint8_t*>(c->d_ref_der.p) + off[l];
      a.cur_img[l] = c->chain ? a.ref_img[l] + a.stride[l] : static_cast<uint8_t*>(c->d_cur_der.p) + off[l];
    }
    c->der_src = src, c->der_top = max_level;
  }
  if (in_kernel) {  // the persistent alignment kernel derives the levels pair by pair (gated host pipeline)
    a.derive_from = src;
    return PLSVO_OK;
  }
  if (b1 <= b0) return PLSVO_OK;
  // frame chain: one stack; pairs [b0,b1) need frames [b0, b1], of which frame b0 was derived with the previous range
  const size_t f0 = c->chain ? (b0 ? b0 + 1 : 0) : b0, f1 = c->chain ? b1 + 1 : b1;
  for (int which = 0; which < (c->chain ? 1 : 2); ++which) {
    PyramidArgs pa;
    memset(&pa, 0, sizeof pa);
    pa.B = (int)(f1 - f0), pa.width = a.width >> src, pa.height = a.height >> src, pa.n_levels = max_level - src + 1;
    for (int l = src; l <= max_level; ++l) {
      const uint8_t* base = which ? a.cur_img[l] : a.ref_img[l];
      pa.level[l - src] = const_cast<uint8_t*>(base) + f0 * a.stride[l];
      pa.pitch[l - src] = a.pitch[l];
      pa.stride[l - src] = a.stride[l];
    }
    // the kernel indexes images with blockIdx.z
    for (int z0 = 0; z0 < pa.B; z0 += 32768) {
      PyramidArgs q = pa;
      q.B = std::min(32768, pa.B - z0);
      for (int k = 0; k < pa.n_levels; ++k) q.level[k] = pa.level[k] + (size_t)z0 * pa.stride[k];
      CK(pyramid_kernel_launch(q, s));
    }
    c->launches += 1;
  }
  return PLSVO_OK;
}

// launch plan of the alignment kernel for the uploaded batch (shared memory, CTA size, grid)
struct AlignPlan {
  int threads, min_blocks, ctas_per_sm;
  size_t smem;
};

// kernel variants (threads per CTA, resident CTAs per SM the register budget is compiled for), see align_kernel.cu
static const int kAlignVariants[][2] = {{128, 4}, {128, 5}, {96, 5}, {96, 7}, {64, 8}, {160, 3}, {192, 2}, {256, 2}};

int align_plan(plsvo_ctx_impl* c, const plsvo_align_params* p, int chunk_pairs, AlignPlan* plan, bool streamed = false) {
  if (!c->align_ready) return fail(c, PLSVO_ERR_STATE, "plsvo_align_launch before plsvo_align_upload");
  if (p->min_level < 0 || p->max_level < p->min_level || p->max_level >= PLSVO_MAX_LEVELS || p->n_iter < 1)
    return fail(c, PLSVO_ERR_INVALID, "level range / n_iter");
  AlignArgs& a = c->aa;
  for (int l = p->min_level; l <= p->max_level; ++l)
    if (!a.pitch[l] || !a.ref_img[l])
      return fail(c, PLSVO_ERR_INVALID, "a pyramid level in [min_level,max_level] was neither uploaded nor derived");
  CK(cudaSetDevice(c->device));
  a.max_level = p->max_level, a.min_level = p->min_level, a.n_iter = p->n_iter, a.eps = p->eps;
  a.max_seg_patches = std::max(c->seg_patch_bound[p->min_level], 1);
  a.max_seg_slots = (c->seg_slot_bound[p->min_level] + 31) / 32 * 32 + 32;
  if (a.max_seg_slots > 65504) return fail(c, PLSVO_ERR_INVALID, "segment samples exceed the lane-slot plan");
  a.max_patches = (a.n_pts + a.max_seg_patches + 3) / 4 * 4;
  if (a.max_patches == 0) a.max_patches = 4;
  const int maxN = std::max(c->seg_maxN[p->min_level], 1);

  // Kernel variant.  Default: 128-thread CTAs with the register budget of four resident pairs per SM; small
  // batches (at most one pair per SM) take 256-thread CTAs to cut the latency of a pair.
  // PLSVO_VARIANT="threads,ctas" selects another compiled variant (tuning / the A-B runs in profiles/).
  int want_t = 128, want_b = 4;
  if (chunk_pairs <= c->num_sms) want_t = 256, want_b = 2;
  // streamed host path: pairs trickle in at the rate of the host link, so fewer are in flight than the grid has room for
  // and the call ends one pair-latency after the last chunk lands — bigger CTAs shorten that tail (tools/e2e_trace.py)
  else if (streamed) want_t = 192, want_b = 2;
  if (const char* v = getenv("PLSVO_VARIANT")) {
    int t = 0, mb = 0;
    if (sscanf(v, "%d,%d", &t, &mb) == 2) {
      bool known = false;
      for (auto& kv : kAlignVariants) known |= (kv[0] == t && kv[1] == mb);
      if (!known) return fail(c, PLSVO_ERR_INVALID, "PLSVO_VARIANT names a variant that is not compiled");
      want_t = t, want_b = mb;
    }
  }
  const int limit = c->smem_optin;  // 227 KB on sm_100a
  // try the wanted variant first, then bigger CTAs (more patches per round, fewer records per thread)
  const int order[][2] = {{want_t, want_b}, {128, 4}, {256, 2}};
  int rc_last = PLSVO_ERR_INVALID;
  for (auto& v : order) {
    const int threads = v[0], min_blocks = v[1];
    // parked in-patch sums of a segment longer than a warp (one record per thread and 32-sample trip)
    const int rec_cap = std::max(1, (maxN + 31) / 32);
    if (rec_cap > 32) {
      rc_last = fail(c, PLSVO_ERR_INVALID, "a segment has more than 1024 samples");
      continue;
    }
    // shared-memory plan: stage the current image level when the CTA still fits min_blocks times per SM next to
    // the per-pair state; bigger levels are read through L2 with the same aligned-word loads.
    const int other = (int)align_smem_bytes(a.n_pts, a.n_segs, a.max_patches, a.max_seg_slots, 0, threads);
    int img_budget = (limit + 1024) / min_blocks - 1024 - other;
    if (img_budget < 0) img_budget = 0;
    img_budget = std::min(img_budget, 96 * 1024);
    if (const char* e = getenv("PLSVO_IMG_SMEM")) img_budget = atoi(e) ? 96 * 1024 : 0;
    int img_bytes = 0;
    for (int l = 0; l < PLSVO_MAX_LEVELS; ++l) a.img_in_smem[l] = 0;
    for (int l = p->min_level; l <= p->max_level; ++l) {
      const size_t bytes = a.stride[l];
      a.img_in_smem[l] = (bytes <= (size_t)img_budget && bytes < (1u << 20) && bytes % 16 == 0) ? 1 : 0;
      if (a.img_in_smem[l]) img_bytes = std::max(img_bytes, (int)bytes);
    }
    size_t smem = align_smem_bytes(a.n_pts, a.n_segs, a.max_patches, a.max_seg_slots, img_bytes, threads);
    if (smem > (size_t)limit) {  // drop image staging as a last resort
      for (int l = 0; l < PLSVO_MAX_LEVELS; ++l) a.img_in_smem[l] = 0;
      img_bytes = 0;
      smem = align_smem_bytes(a.n_pts, a.n_segs, a.max_patches, a.max_seg_slots, 0, threads);
      if (smem > (size_t)limit) {
        rc_last = fail(c, PLSVO_ERR_INVALID, "feature counts exceed the shared-memory plan");
        continue;
      }
    }
    a.smem_img_bytes = img_bytes;
    a.rec_cap = rec_cap;
    a.one = 1.0f;
    int ctas_per_sm = 0;
    CK(align_kernel_prepare(threads, min_blocks, smem, &ctas_per_sm));
    if (ctas_per_sm < 1) {
      rc_last = fail(c, PLSVO_ERR_INVALID, "kernel does not fit on an SM");
      continue;
    }
    const char* cap = getenv("PLSVO_CTAS_PER_SM");
    if (cap && atoi(cap) > 0) ctas_per_sm = std::min(ctas_per_sm, atoi(cap));
    // per-CTA workspaces (L2 resident): reference-patch cache, patch geometry, segment sample centres, pass records
    const size_t grid_max = (size_t)std::min(a.B, c->num_sms * ctas_per_sm);
    CK(ensure(c->d_ws_cache, grid_max * kCacheRows * a.max_patches * sizeof(float4)));
    CK(ensure(c->d_ws_segpx, grid_max * 2 * a.max_seg_patches * sizeof(double)));
    CK(ensure(c->d_ws_rec, grid_max * 5 * (size_t)rec_cap * threads * sizeof(double)));
    a.ws_cache = static_cast<float4*>(c->d_ws_cache.p);
    a.ws_segpx = static_cast<double*>(c->d_ws_segpx.p);
    a.ws_rec = static_cast<double*>(c->d_ws_rec.p);
    plan->threads = threads, plan->min_blocks = min_blocks, plan->ctas_per_sm = ctas_per_sm, plan->smem = smem;
    return PLSVO_OK;
  }
  return rc_last;
}

// one kernel over pairs [b0,b1) of the uploaded batch (pointers rebased to the chunk).  units_ok: the whole batch in one
// ungated launch, where the work queue may hand out (pair, level) units (see below).
int align_launch_range(plsvo_ctx_impl* c, const AlignPlan& plan, size_t b0, size_t b1, int counter_slot, cudaStream_t s,
                       int gate_chunk = 0, bool units_ok = false) {
  AlignArgs a = c->aa;
  const size_t np = (size_t)a.n_pts, ns = (size_t)a.n_segs;
  a.B = (int)(b1 - b0);
  for (int l = 0; l < PLSVO_MAX_LEVELS; ++l) {
    if (!a.pitch[l]) continue;
    a.ref_img[l] += b0 * a.stride[l];
    a.cur_img[l] += b0 * a.stride[l];
  }
#define REBASE(f, per) \
  if (a.f) a.f += b0 * (per)
  REBASE(T_ref_w, 7);
  REBASE(T_cur_w, 7);
  REBASE(pt_count, 1);
  REBASE(pt_px, np * 2);
  REBASE(pt_f, np * 3);
  REBASE(pt_pos, np * 3);
  REBASE(pt_valid, np);
  REBASE(seg_count, 1);
  REBASE(seg_spx, ns * 2);
  REBASE(seg_epx, ns * 2);
  REBASE(seg_sf, ns * 3);
  REBASE(seg_ef, ns * 3);
  REBASE(seg_spos, ns * 3);
  REBASE(seg_epos, ns * 3);
  REBASE(seg_length, ns);
  REBASE(seg_valid, ns);
  REBASE(pt_depth, np);
  REBASE(seg_sdepth, ns);
  REBASE(seg_edepth, ns);
  REBASE(out_T, 7);
  REBASE(out_n_tracked, 1);
  REBASE(out_H, 36);
  REBASE(out_seg_killed, ns);
  REBASE(out_iters, PLSVO_MAX_LEVELS);
  REBASE(out_status, 1);
  REBASE(out_patch_iters, 1);
  REBASE(out_patch_levels, 1);
#undef REBASE
  a.work_counter = c->aa.work_counter + counter_slot;
  a.arrived = gate_chunk > 0 ? c->aa.work_counter + 32 : nullptr;
  a.gate_chunk = gate_chunk;
  const int slots = c->num_sms * plan.ctas_per_sm;
  const int grid = std::min(a.B, slots);
  // Level units: a persistent slot that owns a whole pair idles once the queue is empty while the slowest pairs of the
  // second wave finish.  When the batch has more pairs than the grid has slots, the queue hands out (pair, level) units
  // instead — same CTA shape, same arithmetic, bit-identical results — so the ragged end shrinks to a fraction of a pair.
  // Not on the arrival-gated path (pairs trickle in) nor with levels the kernel derives itself.
  // PLSVO_ALIGN_SCHEDULE=pair|level forces either mode (A/B runs, tests).
  bool units = units_ok && gate_chunk == 0 && a.derive_from < 0 && a.max_level > a.min_level && a.B > slots;
  if (const char* e = getenv("PLSVO_ALIGN_SCHEDULE")) {
    if (!strcmp(e, "pair")) units = false;
    else if (!strcmp(e, "level")) units = units_ok && gate_chunk == 0 && a.derive_from < 0;
  }
  a.level_units = units ? 1 : 0;
  if (units) {
    const size_t done_bytes = (size_t)a.B * sizeof(unsigned long long);
    if (c->d_unit_done.cap < done_bytes) {  // fresh words must not match any epoch
      CK(ensure(c->d_unit_done, done_bytes));
      CK(cudaMemsetAsync(c->d_unit_done.p, 0, c->d_unit_done.cap, s));
    }
    a.unit_state_stride = align_unit_state_stride(a.n_pts, a.n_segs);
    CK(ensure(c->d_unit_state, (size_t)a.B * a.unit_state_stride));
    a.unit_done = static_cast<unsigned long long*>(c->d_unit_done.p);
    a.unit_state = static_cast<unsigned char*>(c->d_unit_state.p);
    a.unit_epoch = ++c->unit_epoch;
  }
  CK(cudaMemsetAsync(a.work_counter, 0, sizeof(unsigned int), s));
  CK(align_kernel_launch(a, grid, plan.threads, plan.min_blocks, plan.smem, s));
  c->launches += 1;
  return PLSVO_OK;
}

}  // namespace

extern "C" {

int plsvo_align_upload(plsvo_ctx* ctx, const plsvo_align_batch* h) {
  if (!ctx || !h) return PLSVO_ERR_INVALID;
  plsvo_ctx_impl* c = CTX(ctx);
  return align_upload_impl(c, h, 0, (size_t)std::max(h->batch, 0), c->stream, 1);
}

int plsvo_align_launch(plsvo_ctx* ctx, const plsvo_align_params* p) {
  if (!ctx || !p) return PLSVO_ERR_INVALID;
  plsvo_ctx_impl* c = CTX(ctx);
  if (!c->align_ready) return fail(c, PLSVO_ERR_STATE, "plsvo_align_launch before plsvo_align_upload");
  if (p->min_level < 0 || p->max_level < p->min_level || p->max_level >= PLSVO_MAX_LEVELS)
    return fail(c, PLSVO_ERR_INVALID, "level range / n_iter");
  AlignPlan plan;
  int rc = align_derive_levels(c, p->min_level, p->max_level, 0, (size_t)c->aa.B, c->stream, false);
  if (rc != PLSVO_OK) return rc;
  rc = align_plan(c, p, c->aa.B, &plan);
  if (rc != PLSVO_OK) return rc;
  return align_launch_range(c, plan, 0, (size_t)c->aa.B, 0, c->stream, 0, /*units_ok=*/true);
}

int plsvo_align_download(plsvo_ctx* ctx, const plsvo_align_result* o) {
  if (!ctx || !o) return PLSVO_ERR_INVALID;
  plsvo_ctx_impl* c = CTX(ctx);
  if (!c->align_ready) return fail(c, PLSVO_ERR_STATE, "plsvo_align_download before plsvo_align_upload");
  CK(cudaSetDevice(c->device));
  const AlignArgs& a = c->aa;
  const size_t B = (size_t)a.B;
  cudaStream_t s = c->stream;
  // one D2H of the whole output block into pinned staging, then plain copies into the caller's arrays
  // (which are usually pageable: eight separate device->pageable copies cost several times more)
  CK(cudaMemcpyAsync(c->h_out, c->d_out_T.p, c->out_bytes, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  const char* hb = c->h_out;
  if (o->T_cur_w) memcpy(o->T_cur_w, hb + c->oo_T, B * 7 * sizeof(double));
  if (o->n_tracked) memcpy(o->n_tracked, hb + c->oo_ntr, B * sizeof(int64_t));
  if (o->H) memcpy(o->H, hb + c->oo_H, B * 36 * sizeof(double));
  if (o->seg_killed && a.n_segs > 0) memcpy(o->seg_killed, hb + c->oo_killed, B * a.n_segs);
  if (o->iters) memcpy(o->iters, hb + c->oo_iters, B * PLSVO_MAX_LEVELS * sizeof(int32_t));
  if (o->status) memcpy(o->status, hb + c->oo_status, B * sizeof(int32_t));
  if (o->patch_iters) memcpy(o->patch_iters, hb + c->oo_pi, B * sizeof(uint32_t));
  if (o->patch_levels) memcpy(o->patch_levels, hb + c->oo_pl, B * sizeof(uint32_t));
  return PLSVO_OK;
}

static int align_batch_run_body(plsvo_ctx* ctx, const plsvo_align_batch* b, const plsvo_align_params* p,
                                const plsvo_align_result* o) {
  plsvo_ctx_impl* c = CTX(ctx);
  // Host-buffer pipeline.  Default for large batches: ONE persistent kernel over the whole batch is
  // launched immediately while a second stream copies the batch to the device in chunks of 256 pairs
  // and bumps an arrival counter after each chunk; the kernel's work queue hands a pair out only once
  // its chunk has landed (arrival gate), so the PCIe leg and the compute leg overlap without cutting
  // the batch into under-filled kernels.  Chunks of 128 pairs keep every array's chunk boundary
  // 128-byte aligned (no cache line shared between an arrived and an in-flight chunk).
  // PLSVO_E2E_CHUNKS=k (k>=2) selects the older k-kernel pipeline, PLSVO_E2E_CHUNKS=1 the plain
  // upload -> launch -> download sequence.
  int chunks = 0;
  const char* cenv = getenv("PLSVO_E2E_CHUNKS");
  if (cenv && atoi(cenv) >= 1) chunks = std::min(atoi(cenv), 8);
  bool gated = (chunks == 0) && b->batch >= 256;
  if (gated) {
    for (int l = p->min_level; l <= p->max_level && l < PLSVO_MAX_LEVELS && l >= 0; ++l) {
      const int rows = b->cam.height >> l;
      if (!b->ref_img[l] && l > p->min_level) continue;  // derived on the device after each chunk has landed
      const bool direct = b->ref_img[l] && b->img_stride[l] == (size_t)rows * b->img_pitch[l] && b->img_pitch[l] % 4 == 0 &&
                          b->img_stride[l] % 16 == 0;
      if (!direct) gated = false;  // padded layouts need a device-side repack kernel: not under the gate
      // frame chain: the last frame of an arrived chunk and the first frame of the chunk in flight are neighbours in one
      // stack — they must not share a 128-byte line
      if ((b->flags & PLSVO_ALIGN_FRAME_CHAIN) && b->img_stride[l] % 128 != 0) gated = false;
    }
  }
  if (gated) {
    CK(cudaSetDevice(c->device));
    if (!c->copy_stream) {
      CK(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
      for (int k = 0; k < 8; ++k) CK(cudaEventCreateWithFlags(&c->chunk_ev[k], cudaEventDisableTiming));
      CK(cudaEventCreateWithFlags(&c->start_ev, cudaEventDisableTiming));
    }
    const size_t B = (size_t)b->batch;
    int chunk = 256;  // multiple of 128 pairs: every array's chunk boundary stays 128-byte aligned (tools/tune_e2e.py)
    const char* genv = getenv("PLSVO_GATE_CHUNK");
    if (genv && atoi(genv) >= 128) chunk = atoi(genv) / 128 * 128;
    const int n_chunks = (int)((B + chunk - 1) / chunk);
    if (!c->h_flags || c->h_flags_cap < n_chunks) {
      if (c->h_flags) cudaFreeHost(c->h_flags);
      c->h_flags = nullptr;
      CK(cudaHostAlloc((void**)&c->h_flags, sizeof(unsigned int) * (size_t)n_chunks, cudaHostAllocDefault));
      c->h_flags_cap = n_chunks;
    }
    for (int k = 0; k < n_chunks; ++k) c->h_flags[k] = (unsigned int)(k + 1);
    // the copy stream must not overtake work already queued on the main stream; the arrival counter is
    // cleared on the main stream before the copy stream may bump it
    CK(ensure(c->d_counter, 256));
    unsigned int* d_arrived = static_cast<unsigned int*>(c->d_counter.p) + 32;
    CK(cudaMemsetAsync(d_arrived, 0, sizeof(unsigned int), c->stream));
    // PLSVO_TRACE_E2E=1: timeline of this call on stderr (chunk arrival times, kernel end, download end) — measurement aid
    const bool trace = getenv("PLSVO_TRACE_E2E") != nullptr;
    cudaEvent_t tr_start = nullptr, tr_chunk[64] = {nullptr}, tr_kernel = nullptr;
    const auto t_host0 = std::chrono::steady_clock::now();
    if (trace) {
      cudaEventCreate(&tr_start), cudaEventCreate(&tr_kernel);
      for (int k = 0; k < n_chunks && k < 64; ++k) cudaEventCreate(&tr_chunk[k]);
      cudaEventRecord(tr_start, c->stream);
    }
    CK(cudaEventRecord(c->start_ev, c->stream));
    CK(cudaStreamWaitEvent(c->copy_stream, c->start_ev, 0));
    // extra copy streams (PLSVO_COPY_STREAMS, default 1 = the copy stream alone): a chunk's ~24 array copies go
    // round-robin over them and the arrival flag waits for all of them
    int n_rr = 1;
    const char* renv = getenv("PLSVO_COPY_STREAMS");
    if (renv && atoi(renv) >= 1) n_rr = std::min(atoi(renv), 4);
    if (n_rr > 1) {
      for (int k = 0; k < n_rr; ++k) {
        if (!c->rr_stream[k]) {
          CK(cudaStreamCreateWithFlags(&c->rr_stream[k], cudaStreamNonBlocking));
          CK(cudaEventCreateWithFlags(&c->rr_ev[k], cudaEventDisableTiming));
        }
        CK(cudaStreamWaitEvent(c->rr_stream[k], c->start_ev, 0));
      }
    }
    // enqueue every chunk copy first (asynchronous from pinned memory): the host-side sizing below and
    // the kernel launch then overlap with the DMA
    int rc = PLSVO_OK;
    // every feature array of the whole batch first (a dozen large copies, ~a quarter of the bytes), then the images chunk
    // by chunk (two copies per chunk and level): few, large transfers keep the link near its peak rate and the arrival
    // flags then track the image stream alone.  PLSVO_GATE_INTERLEAVED=1 restores the per-chunk slices of every array.
    const bool features_first = !getenv("PLSVO_GATE_INTERLEAVED");
    if (features_first) {
      rc = align_upload_impl(c, b, 0, B, c->copy_stream, 2, /*what=*/2);
      if (rc != PLSVO_OK) {
        cudaStreamSynchronize(c->copy_stream);
        return rc;
      }
    }
    for (int k = 0; k < n_chunks; ++k) {
      c->rr_n = n_rr > 1 ? n_rr : 0, c->rr_i = 0;
      rc = align_upload_impl(c, b, (size_t)k * chunk, std::min<size_t>((size_t)(k + 1) * chunk, B), c->copy_stream,
                             (k == 0 && !features_first) ? 2 : 0, features_first ? 1 : 3);
      c->rr_n = 0;
      if (rc != PLSVO_OK) {
        cudaStreamSynchronize(c->copy_stream);
        return rc;
      }
      for (int j = 0; j < (n_rr > 1 ? n_rr : 0); ++j) {
        CK(cudaEventRecord(c->rr_ev[j], c->rr_stream[j]));
        CK(cudaStreamWaitEvent(c->copy_stream, c->rr_ev[j], 0));
      }
      // coarser levels that were not shipped: the persistent kernel halfSamples them pair by pair (a pyramid kernel
      // behind this chunk's copies could not become resident next to the grid that waits for it)
      rc = align_derive_levels(c, p->min_level, p->max_level, (size_t)k * chunk, std::min<size_t>((size_t)(k + 1) * chunk, B), c->copy_stream,
                               k == 0, /*in_kernel=*/true);
      if (rc != PLSVO_OK) {
        cudaStreamSynchronize(c->copy_stream);  // the caller's host arrays must not be read after we return
        return rc;
      }
      CK(cudaMemcpyAsync(d_arrived, &c->h_flags[k], sizeof(unsigned int), cudaMemcpyHostToDevice, c->copy_stream));
      if (trace && k < 64) cudaEventRecord(tr_chunk[k], c->copy_stream);
    }
    const auto t_host1 = std::chrono::steady_clock::now();
    // host-side sizing (segment-sample bound of the finest level, outputs): on the launch path, so the cheap bound
    rc = align_upload_impl(c, b, 0, 0, c->copy_stream, 3, 3, getenv("PLSVO_EXACT_SIZING") ? -1 : p->min_level);
    AlignPlan plan;
    if (rc == PLSVO_OK) rc = align_plan(c, p, (int)B, &plan, /*streamed=*/true);
    if (rc != PLSVO_OK) {
      // copies are in flight: the caller's host arrays must not be read after we return
      cudaStreamSynchronize(c->copy_stream);
      for (int j = 0; j < 4; ++j)
        if (c->rr_stream[j]) cudaStreamSynchronize(c->rr_stream[j]);
      return rc;
    }
    const auto t_host2 = std::chrono::steady_clock::now();
    rc = align_launch_range(c, plan, 0, B, 0, c->stream, chunk);  // gated on arrivals
    if (rc != PLSVO_OK) return rc;
    if (trace) cudaEventRecord(tr_kernel, c->stream);
    const auto t_host3 = std::chrono::steady_clock::now();
    rc = plsvo_align_download(ctx, o);
    if (trace) {
      const auto t_host4 = std::chrono::steady_clock::now();
      auto ms = [&](std::chrono::steady_clock::time_point t) { return std::chrono::duration<double, std::milli>(t - t_host0).count(); };
      std::fprintf(stderr, "[plsvo e2e trace] host: copies enqueued %.3f, sized+planned %.3f, launched %.3f, returned %.3f ms | device:", ms(t_host1),
                   ms(t_host2), ms(t_host3), ms(t_host4));
      for (int k = 0; k < n_chunks && k < 64; ++k) {
        float t = 0;
        cudaEventElapsedTime(&t, tr_start, tr_chunk[k]);
        std::fprintf(stderr, " chunk%d %.3f", k, t);
        cudaEventDestroy(tr_chunk[k]);
      }
      float t = 0;
      cudaEventElapsedTime(&t, tr_start, tr_kernel);
      std::fprintf(stderr, " kernel_end %.3f ms\n", t);
      cudaEventDestroy(tr_start), cudaEventDestroy(tr_kernel);
    }
    return rc;
  }
  if (chunks == 0) chunks = 1;
  if (chunks > b->batch) chunks = 1;
  if (chunks == 1) {
    int rc = plsvo_align_upload(ctx, b);
    if (rc != PLSVO_OK) return rc;
    rc = plsvo_align_launch(ctx, p);
    if (rc != PLSVO_OK) return rc;
    return plsvo_align_download(ctx, o);
  }
  CK(cudaSetDevice(c->device));
  if (!c->copy_stream) {
    CK(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    for (int k = 0; k < 8; ++k) CK(cudaEventCreateWithFlags(&c->chunk_ev[k], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&c->start_ev, cudaEventDisableTiming));
  }
  // the copy stream must not overtake work already queued on the main stream (previous batch's kernels
  // still read the device buffers)
  CK(cudaEventRecord(c->start_ev, c->stream));
  CK(cudaStreamWaitEvent(c->copy_stream, c->start_ev, 0));
  const size_t B = (size_t)b->batch;
  AlignPlan plan;
  for (int k = 0; k < chunks; ++k) {
    const size_t b0 = B * k / chunks, b1 = B * (k + 1) / chunks;
    int rc = align_upload_impl(c, b, b0, b1, c->copy_stream, k == 0 ? 1 : 0);
    if (rc != PLSVO_OK) return rc;
    rc = align_derive_levels(c, p->min_level, p->max_level, b0, b1, c->copy_stream, k == 0);
    if (rc != PLSVO_OK) return rc;
    CK(cudaEventRecord(c->chunk_ev[k], c->copy_stream));
    if (k == 0) {
      rc = align_plan(c, p, (int)(b1 - b0), &plan);
      if (rc != PLSVO_OK) return rc;
    }
    CK(cudaStreamWaitEvent(c->stream, c->chunk_ev[k], 0));
    rc = align_launch_range(c, plan, b0, b1, k, c->stream);
    if (rc != PLSVO_OK) return rc;
  }
  return plsvo_align_download(ctx, o);
}

int plsvo_align_batch_run(plsvo_ctx* ctx, const plsvo_align_batch* b, const plsvo_align_params* p,
                          const plsvo_align_result* o) {
  if (!ctx || !b || !p || !o) return PLSVO_ERR_INVALID;
  return settled(CTX(ctx), align_batch_run_body(ctx, b, p, o));
}

// ------------------------------------------------------------------------------------------------
// pose optimiser
// ------------------------------------------------------------------------------------------------
}  // extern "C"

namespace {
// device_T: poses already on the device (the chained call), instead of h->T_f_w
int poseopt_upload_impl(plsvo_ctx_impl* c, const plsvo_poseopt_batch* h, const double* device_T) {
  c->po_ready = false;
  if (h->batch <= 0 || h->n_pts < 0 || h->n_segs < 0) return fail(c, PLSVO_ERR_INVALID, "batch/n_pts/n_segs out of range");
  if (!h->T_f_w && !device_T) return fail(c, PLSVO_ERR_INVALID, "T_f_w missing");
  for (int b = 0; b < h->batch; ++b) {  // the counts index shared memory in the kernel
    if (h->pt_count && (h->pt_count[b] < 0 || h->pt_count[b] > h->n_pts)) return fail(c, PLSVO_ERR_INVALID, "pt_count[b] outside [0, n_pts]");
    if (h->seg_count && (h->seg_count[b] < 0 || h->seg_count[b] > h->n_segs))
      return fail(c, PLSVO_ERR_INVALID, "seg_count[b] outside [0, n_segs]");
  }
  if (h->n_pts > 0 && (!h->pt_f || !h->pt_pos || !h->pt_level)) return fail(c, PLSVO_ERR_INVALID, "point arrays missing");
  if (h->n_segs > 0 && (!h->seg_line || !h->seg_spos || !h->seg_epos || !h->seg_level))
    return fail(c, PLSVO_ERR_INVALID, "segment arrays missing");
  CK(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  PoseOptArgs& a = c->pa;
  const size_t B = (size_t)h->batch;
  a.B = h->batch, a.n_pts = h->n_pts, a.n_segs = h->n_segs, a.fx = h->fx;
  {
    const size_t np_ = (size_t)h->n_pts, ns_ = (size_t)h->n_segs;
    struct Item {
      const void* host;
      size_t bytes;
      const void** dev;
      DevBuf* buf;
    };
    const Item items[] = {
        {device_T ? nullptr : h->T_f_w, B * 7 * 8, (const void**)&a.T_f_w, &c->p_T},
        {h->pt_count, B * 4, (const void**)&a.pt_count, &c->p_pt_count},
        {h->pt_f, B * np_ * 24, (const void**)&a.pt_f, &c->p_pt_f},
        {h->pt_pos, B * np_ * 24, (const void**)&a.pt_pos, &c->p_pt_pos},
        {h->pt_level, B * np_ * 4, (const void**)&a.pt_level, &c->p_pt_level},
        {h->pt_valid, B * np_, (const void**)&a.pt_valid, &c->p_pt_valid},
        {h->seg_count, B * 4, (const void**)&a.seg_count, &c->p_seg_count},
        {h->seg_line, B * ns_ * 24, (const void**)&a.seg_line, &c->p_seg_line},
        {h->seg_spos, B * ns_ * 24, (const void**)&a.seg_spos, &c->p_seg_spos},
        {h->seg_epos, B * ns_ * 24, (const void**)&a.seg_epos, &c->p_seg_epos},
        {h->seg_level, B * ns_ * 4, (const void**)&a.seg_level, &c->p_seg_level},
        {h->seg_valid, B * ns_, (const void**)&a.seg_valid, &c->p_seg_valid},
    };
    size_t total = 0;
    for (const Item& it : items)
      if (it.host && it.bytes) total += (it.bytes + 255) / 256 * 256;
    // small batches (the reference's own call is one frame, frame_handler_mono.cpp:327-329): every input packed into one
    // pinned block and moved with ONE copy instead of a dozen staged pageable ones
    const bool small = total > 0 && total <= ((size_t)4 << 20) && !getenv("PLSVO_NO_SMALL_UPLOAD");
    if (small) {
      if (c->h_in_cap < total + 256) {
        if (c->h_in_ev) CK(cudaEventSynchronize(c->h_in_ev));
        if (c->h_in) cudaFreeHost(c->h_in);
        c->h_in = nullptr, c->h_in_cap = 0;
        CK(cudaHostAlloc((void**)&c->h_in, total + 256, cudaHostAllocDefault));
        c->h_in_cap = total + 256;
      }
      if (!c->h_in_ev) CK(cudaEventCreateWithFlags(&c->h_in_ev, cudaEventDisableTiming));
      else CK(cudaEventSynchronize(c->h_in_ev));  // the previous packed upload has left the staging block
      CK(ensure(c->p_in, total + 256));
      size_t off = 0;
      for (const Item& it : items) {
        if (!it.host || !it.bytes) {
          if (!(it.dev == (const void**)&a.T_f_w && device_T)) *it.dev = nullptr;
          continue;
        }
        memcpy(c->h_in + off, it.host, it.bytes);
        *it.dev = static_cast<char*>(c->p_in.p) + off;
        off += (it.bytes + 255) / 256 * 256;
      }
      CK(cudaMemcpyAsync(c->p_in.p, c->h_in, total, cudaMemcpyHostToDevice, s));
      CK(cudaEventRecord(c->h_in_ev, s));
    } else {
      for (const Item& it : items) {
        if (!it.host || !it.bytes) {
          if (!(it.dev == (const void**)&a.T_f_w && device_T)) *it.dev = nullptr;
          continue;
        }
        CK(ensure(*it.buf, it.bytes));
        *it.dev = it.buf->p;
        CK(cudaMemcpyAsync(it.buf->p, it.host, it.bytes, cudaMemcpyHostToDevice, s));
      }
    }
    if (device_T) a.T_f_w = device_T;
  }
  // all outputs live in one device block: cleared with one memset where the kernel may leave them untouched, and brought
  // back with a single D2H into pinned staging
  {
    size_t o = 0;
    auto take = [&](size_t bytes) {
      const size_t at = o;
      o = (o + bytes + 255) / 256 * 256;
      return at;
    };
    const size_t oT = take(B * 7 * sizeof(double));
    const size_t ocov = take(B * 36 * sizeof(double)), oscale = take(B * sizeof(double)), oei = take(B * sizeof(double));
    const size_t oef = take(B * sizeof(double)), onpt = take(B * sizeof(long long)), onls = take(B * sizeof(long long));
    const size_t zero_end = o;
    const size_t opto = take(B * (size_t)std::max(1, h->n_pts)), osgo = take(B * (size_t)std::max(1, h->n_segs));
    const size_t oit = take(B * 2 * sizeof(int32_t)), ost = take(B * sizeof(int32_t));
    c->po_out_bytes = o, c->po_zero_off = ocov, c->po_zero_bytes = zero_end - ocov;
    CK(ensure(c->p_out_T, o));
    if (c->h_po_out_cap < o) {
      if (c->h_po_out) cudaFreeHost(c->h_po_out);
      c->h_po_out = nullptr, c->h_po_out_cap = 0;
      CK(cudaHostAlloc((void**)&c->h_po_out, o, cudaHostAllocDefault));
      c->h_po_out_cap = o;
    }
    char* base = static_cast<char*>(c->p_out_T.p);
    a.out_T = reinterpret_cast<double*>(base + oT);
    a.out_cov = reinterpret_cast<double*>(base + ocov);
    a.out_scale = reinterpret_cast<double*>(base + oscale);
    a.out_err_init = reinterpret_cast<double*>(base + oei);
    a.out_err_final = reinterpret_cast<double*>(base + oef);
    a.out_num_pt = reinterpret_cast<long long*>(base + onpt);
    a.out_num_ls = reinterpret_cast<long long*>(base + onls);
    a.out_pt_outlier = reinterpret_cast<uint8_t*>(base + opto);
    a.out_seg_outlier = reinterpret_cast<uint8_t*>(base + osgo);
    a.out_iters = reinterpret_cast<int32_t*>(base + oit);
    a.out_status = reinterpret_cast<int32_t*>(base + ost);
  }
  c->po_ready = true;
  return PLSVO_OK;
}
}  // namespace

extern "C" {

int plsvo_poseopt_upload(plsvo_ctx* ctx, const plsvo_poseopt_batch* h) {
  if (!ctx || !h) return PLSVO_ERR_INVALID;
  return poseopt_upload_impl(CTX(ctx), h, nullptr);
}

int plsvo_poseopt_launch(plsvo_ctx* ctx, const plsvo_poseopt_params* p) {
  if (!ctx || !p) return PLSVO_ERR_INVALID;
  plsvo_ctx_impl* c = CTX(ctx);
  if (!c->po_ready) return fail(c, PLSVO_ERR_STATE, "plsvo_poseopt_launch before plsvo_poseopt_upload");
  if (p->n_iter < 0) return fail(c, PLSVO_ERR_INVALID, "n_iter");
  CK(cudaSetDevice(c->device));
  PoseOptArgs& a = c->pa;
  a.reproj_thresh = p->reproj_thresh, a.n_iter = p->n_iter, a.n_iter_ref = p->n_iter_ref;
  const size_t smem = poseopt_smem_bytes(a.n_pts, a.n_segs);
  if (smem > (size_t)c->smem_optin) return fail(c, PLSVO_ERR_INVALID, "feature counts exceed shared memory");
  // outputs of frames that return early keep their previous contents: clear the ones we always report
  CK(cudaMemsetAsync(static_cast<char*>(c->p_out_T.p) + c->po_zero_off, 0, c->po_zero_bytes, c->stream));
  CK(poseopt_kernel_launch(a, smem, c->stream));
  c->launches += 1;
  return PLSVO_OK;
}

int plsvo_poseopt_download(plsvo_ctx* ctx, const plsvo_poseopt_result* o) {
  if (!ctx || !o) return PLSVO_ERR_INVALID;
  plsvo_ctx_impl* c = CTX(ctx);
  if (!c->po_ready) return fail(c, PLSVO_ERR_STATE, "plsvo_poseopt_download before plsvo_poseopt_upload");
  CK(cudaSetDevice(c->device));
  const PoseOptArgs& a = c->pa;
  const size_t B = (size_t)a.B;
  cudaStream_t s = c->stream;
  CK(cudaMemcpyAsync(c->h_po_out, c->p_out_T.p, c->po_out_bytes, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  {
    const char* dbase = static_cast<const char*>(c->p_out_T.p);
    auto host_of = [&](const void* dev) { return c->h_po_out + (static_cast<const char*>(dev) - dbase); };
    if (o->T_f_w) memcpy(o->T_f_w, host_of(a.out_T), B * 7 * sizeof(double));
    if (o->cov) memcpy(o->cov, host_of(a.out_cov), B * 36 * sizeof(double));
    if (o->estimated_scale) memcpy(o->estimated_scale, host_of(a.out_scale), B * sizeof(double));
    if (o->error_init) memcpy(o->error_init, host_of(a.out_err_init), B * sizeof(double));
    if (o->error_final) memcpy(o->error_final, host_of(a.out_err_final), B * sizeof(double));
    if (o->num_obs_pt) memcpy(o->num_obs_pt, host_of(a.out_num_pt), B * sizeof(int64_t));
    if (o->num_obs_ls) memcpy(o->num_obs_ls, host_of(a.out_num_ls), B * sizeof(int64_t));
    if (o->pt_outlier && a.n_pts > 0) memcpy(o->pt_outlier, host_of(a.out_pt_outlier), B * (size_t)a.n_pts);
    if (o->seg_outlier && a.n_segs > 0) memcpy(o->seg_outlier, host_of(a.out_seg_outlier), B * (size_t)a.n_segs);
    if (o->iters) memcpy(o->iters, host_of(a.out_iters), B * 2 * sizeof(int32_t));
    if (o->status) memcpy(o->status, host_of(a.out_status), B * sizeof(int32_t));
  }
  return PLSVO_OK;
}

// FrameHandlerMono::processFrame's two hot-path calls back to back (src/frame_handler_mono.cpp:272-274 and :327-329) for
// a batch of frames, without the pose leaving the device: sparse image alignment of (ref, cur), then the pose optimiser
// on cur's matched features starting from the aligned pose.  pb->T_f_w may be NULL (the usual case): frame b of the
// pose-optimiser batch then starts from the alignment result of pair b, read on the device.
int plsvo_track_upload(plsvo_ctx* ctx, const plsvo_align_batch* ab, const plsvo_poseopt_batch* pb) {
  if (!ctx || !ab || !pb) return PLSVO_ERR_INVALID;
  plsvo_ctx_impl* c = CTX(ctx);
  if (pb->batch != ab->batch) return fail(c, PLSVO_ERR_INVALID, "alignment and pose-optimiser batches differ in size");
  int rc = plsvo_align_upload(ctx, ab);
  if (rc != PLSVO_OK) return rc;
  // the pose optimiser reads the aligned poses where the alignment kernel leaves them (unless poses are given)
  return poseopt_upload_impl(c, pb, pb->T_f_w ? nullptr : c->aa.out_T);
}

int plsvo_track_launch(plsvo_ctx* ctx, const plsvo_align_params* ap, const plsvo_poseopt_params* pp) {
  if (!ctx || !ap || !pp) return PLSVO_ERR_INVALID;
  int rc = plsvo_align_launch(ctx, ap);  // the two kernels back to back on the context's stream
  if (rc != PLSVO_OK) return rc;
  return plsvo_poseopt_launch(ctx, pp);
}

int plsvo_track_batch_run(plsvo_ctx* ctx, const plsvo_align_batch* ab, const plsvo_align_params* ap,
                          const plsvo_poseopt_batch* pb, const plsvo_poseopt_params* pp, const plsvo_align_result* ao,
                          const plsvo_poseopt_result* po) {
  if (!ctx || !ab || !ap || !pb || !pp || !po) return PLSVO_ERR_INVALID;
  int rc = plsvo_track_upload(ctx, ab, pb);
  if (rc == PLSVO_OK) rc = plsvo_track_launch(ctx, ap, pp);
  if (rc == PLSVO_OK && ao) rc = plsvo_align_download(ctx, ao);
  if (rc == PLSVO_OK) rc = plsvo_poseopt_download(ctx, po);
  return settled(CTX(ctx), rc);
}

int plsvo_poseopt_batch_run(plsvo_ctx* ctx, const plsvo_poseopt_batch* b, const plsvo_poseopt_params* p,
                            const plsvo_poseopt_result* o) {
  if (!ctx || !b || !p || !o) return PLSVO_ERR_INVALID;
  int rc = plsvo_poseopt_upload(ctx, b);
  if (rc == PLSVO_OK) rc = plsvo_poseopt_launch(ctx, p);
  if (rc == PLSVO_OK) rc = plsvo_poseopt_download(ctx, o);
  return settled(CTX(ctx), rc);
}

}  // extern "C"

static int pyramid_batch_run_body(plsvo_ctx* ctx, const plsvo_pyramid_batch* in, const plsvo_pyramid_result* out) {
  plsvo_ctx_impl* c = CTX(ctx);
  if (in->batch <= 0 || in->width <= 0 || in->height <= 0 || in->n_levels < 1 || in->n_levels > 7 || !in->img0 ||
      in->pitch0 < (size_t)in->width)
    return fail(c, PLSVO_ERR_INVALID, "pyramid batch description");
  CK(cudaSetDevice(c->device));
  PyramidArgs a;
  memset(&a, 0, sizeof a);
  a.B = in->batch, a.width = in->width, a.height = in->height, a.n_levels = in->n_levels;
  const size_t B = (size_t)in->batch;
  size_t total = 0, off[PLSVO_MAX_LEVELS] = {0};
  for (int l = 0; l < in->n_levels; ++l) {
    const int cols = in->width >> l, rows = in->height >> l;
    if (cols <= 0 || rows <= 0) return fail(c, PLSVO_ERR_INVALID, "pyramid level smaller than one pixel");
    if (l > 0 && !out->level[l]) return fail(c, PLSVO_ERR_INVALID, "output level missing");
    a.pitch[l] = (uint32_t)((cols + 15) / 16 * 16);
    a.stride[l] = (size_t)rows * a.pitch[l];
    total = (total + 255) / 256 * 256;
    off[l] = total;
    total += a.stride[l] * B;
  }
  CK(ensure(c->y_img, total + 256));
  for (int l = 0; l < in->n_levels; ++l) a.level[l] = static_cast<uint8_t*>(c->y_img.p) + off[l];
  cudaStream_t s = c->stream;
  if (in->stride0 == (size_t)in->height * in->pitch0) {
    CK(cudaMemcpy2DAsync(a.level[0], a.pitch[0], in->img0, in->pitch0, in->width, (size_t)in->height * B, cudaMemcpyHostToDevice, s));
  } else {
    for (size_t b = 0; b < B; ++b)
      CK(cudaMemcpy2DAsync(a.level[0] + b * a.stride[0], a.pitch[0], in->img0 + b * in->stride0, in->pitch0, in->width,
                           in->height, cudaMemcpyHostToDevice, s));
  }
  CK(kernel_timer(c, 0, s));
  CK(pyramid_kernel_launch(a, s));
  CK(kernel_timer(c, 1, s));
  c->launches += 1;
  for (int l = 1; l < in->n_levels; ++l) {
    const int cols = in->width >> l, rows = in->height >> l;
    if (out->pitch[l] < (size_t)cols) return fail(c, PLSVO_ERR_INVALID, "output pitch smaller than the level width");
    if (out->stride[l] == (size_t)rows * out->pitch[l]) {
      CK(cudaMemcpy2DAsync(out->level[l], out->pitch[l], a.level[l], a.pitch[l], cols, (size_t)rows * B, cudaMemcpyDeviceToHost, s));
    } else {
      for (size_t b = 0; b < B; ++b)
        CK(cudaMemcpy2DAsync(out->level[l] + b * out->stride[l], out->pitch[l], a.level[l] + b * a.stride[l], a.pitch[l], cols,
                             rows, cudaMemcpyDeviceToHost, s));
    }
  }
  CK(cudaStreamSynchronize(s));
  return PLSVO_OK;
}

namespace {
// align2D (dir == nullptr) and align1D (dir != nullptr) share staging and launch.
int feature_align_run(plsvo_ctx_impl* c, const plsvo_align2d_batch* in, const float* dir, double* o_px, uint8_t* o_conv,
                      double* o_hinv) {
  if (in->n_features < 0 || in->n_images <= 0 || in->width <= 0 || in->height <= 0 || in->n_iter < 0)
    return fail(c, PLSVO_ERR_INVALID, "align2d batch description");
  if (in->n_features == 0) return PLSVO_OK;
  if (!in->image_index || !in->level || !in->ref_patch_with_border || !in->ref_patch || !in->px || !o_px || !o_conv)
    return fail(c, PLSVO_ERR_INVALID, "align2d arrays missing");
  const size_t n = (size_t)in->n_features, B = (size_t)in->n_images;
  for (size_t i = 0; i < n; ++i) {
    const int l = in->level[i];
    if (l < 0 || l >= PLSVO_MAX_LEVELS || !in->img[l] || in->image_index[i] < 0 || in->image_index[i] >= in->n_images)
      return fail(c, PLSVO_ERR_INVALID, "align2d feature refers to a missing level or frame");
  }
  CK(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  Align2DArgs a;
  memset(&a, 0, sizeof a);
  a.n = in->n_features, a.n_iter = in->n_iter, a.width = in->width, a.height = in->height;
  size_t total = 0, off[PLSVO_MAX_LEVELS] = {0};
  for (int l = 0; l < PLSVO_MAX_LEVELS; ++l) {
    if (!in->img[l]) continue;
    const int cols = in->width >> l, rows = in->height >> l;
    if (cols <= 0 || rows <= 0 || in->img_pitch[l] < (size_t)cols) return fail(c, PLSVO_ERR_INVALID, "align2d level geometry");
    a.pitch[l] = (uint32_t)((cols + 15) / 16 * 16);
    a.stride[l] = (size_t)rows * a.pitch[l];
    total = (total + 255) / 256 * 256;
    off[l] = total;
    total += a.stride[l] * B;
  }
  CK(ensure(c->f_img, total + 256));
  for (int l = 0; l < PLSVO_MAX_LEVELS; ++l) {
    if (!in->img[l]) continue;
    const int cols = in->width >> l, rows = in->height >> l;
    uint8_t* d = static_cast<uint8_t*>(c->f_img.p) + off[l];
    a.img[l] = d;
    if (in->img_stride[l] == (size_t)rows * in->img_pitch[l]) {
      CK(cudaMemcpy2DAsync(d, a.pitch[l], in->img[l], in->img_pitch[l], cols, (size_t)rows * B, cudaMemcpyHostToDevice, s));
    } else {
      for (size_t b = 0; b < B; ++b)
        CK(cudaMemcpy2DAsync(d + b * a.stride[l], a.pitch[l], in->img[l] + b * in->img_stride[l], in->img_pitch[l], cols, rows,
                             cudaMemcpyHostToDevice, s));
    }
  }
  CK(up(c->f_idx, in->image_index, n, s, &a.image_index));
  CK(up(c->f_lvl, in->level, n, s, &a.level));
  CK(up(c->f_border, in->ref_patch_with_border, n * 100, s, &a.ref_patch_with_border));
  CK(up(c->f_ref, in->ref_patch, n * 64, s, &a.ref_patch));
  CK(up(c->f_px, in->px, n * 2, s, &a.px));
  CK(ensure(c->f_opx, n * 2 * sizeof(double)));
  CK(ensure(c->f_oconv, n));
  a.out_px = static_cast<double*>(c->f_opx.p);
  a.out_converged = static_cast<uint8_t*>(c->f_oconv.p);
  if (dir) {
    CK(up(c->f_dir, dir, n * 2, s, &a.dir));
    CK(ensure(c->f_ohinv, n * sizeof(double)));
    a.out_h_inv = static_cast<double*>(c->f_ohinv.p);
  }
  CK(kernel_timer(c, 0, s));
  CK(dir ? align1d_kernel_launch(a, s) : align2d_kernel_launch(a, s));
  CK(kernel_timer(c, 1, s));
  c->launches += 1;
  CK(cudaMemcpyAsync(o_px, a.out_px, n * 2 * sizeof(double), cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(o_conv, a.out_converged, n, cudaMemcpyDeviceToHost, s));
  if (dir && o_hinv) CK(cudaMemcpyAsync(o_hinv, a.out_h_inv, n * sizeof(double), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  return PLSVO_OK;
}
}  // namespace

extern "C" int plsvo_align2d_batch_run(plsvo_ctx* ctx, const plsvo_align2d_batch* in, const plsvo_align2d_result* out) {
  if (!ctx || !in || !out) return PLSVO_ERR_INVALID;
  return settled(CTX(ctx), feature_align_run(CTX(ctx), in, nullptr, out->px, out->converged, nullptr));
}

extern "C" int plsvo_align1d_batch_run(plsvo_ctx* ctx, const plsvo_align1d_batch* in, const plsvo_align1d_result* out) {
  if (!ctx || !in || !out) return PLSVO_ERR_INVALID;
  if (in->features.n_features > 0 && !in->dir) return fail(CTX(ctx), PLSVO_ERR_INVALID, "align1d directions missing");
  return settled(CTX(ctx), feature_align_run(CTX(ctx), &in->features, in->dir, out->px, out->converged, out->h_inv));
}

namespace {
// Copies the given pyramid levels of n_images frames to the device with 16-byte row pitch.
int stage_pyramid(plsvo_ctx_impl* c, DevBuf& buf, const uint8_t* const* img, const size_t* pitch, const size_t* stride, int n_images,
                  int width, int height, cudaStream_t s, const uint8_t** d_img, uint32_t* d_pitch, size_t* d_stride) {
  size_t total = 0, off[PLSVO_MAX_LEVELS] = {0};
  const size_t B = (size_t)n_images;
  for (int l = 0; l < PLSVO_MAX_LEVELS; ++l) {
    d_img[l] = nullptr, d_pitch[l] = 0, d_stride[l] = 0;
    if (!img[l]) continue;
    const int cols = width >> l, rows = height >> l;
    if (cols <= 0 || rows <= 0 || pitch[l] < (size_t)cols) return fail(c, PLSVO_ERR_INVALID, "pyramid level geometry");
    d_pitch[l] = (uint32_t)((cols + 15) / 16 * 16);
    d_stride[l] = (size_t)rows * d_pitch[l];
    total = (total + 255) / 256 * 256;
    off[l] = total;
    total += d_stride[l] * B;
  }
  CK(ensure(buf, total + 256));
  for (int l = 0; l < PLSVO_MAX_LEVELS; ++l) {
    if (!img[l]) continue;
    const int cols = width >> l, rows = height >> l;
    uint8_t* d = static_cast<uint8_t*>(buf.p) + off[l];
    d_img[l] = d;
    if (stride[l] == (size_t)rows * pitch[l]) {
      CK(cudaMemcpy2DAsync(d, d_pitch[l], img[l], pitch[l], cols, (size_t)rows * B, cudaMemcpyHostToDevice, s));
    } else {
      for (size_t b = 0; b < B; ++b)
        CK(cudaMemcpy2DAsync(d + b * d_stride[l], d_pitch[l], img[l] + b * stride[l], pitch[l], cols, rows, cudaMemcpyHostToDevice, s));
    }
  }
  return PLSVO_OK;
}
}  // namespace

static int match_direct_batch_run_body(plsvo_ctx* ctx, const plsvo_match_batch* in, const plsvo_match_result* out) {
  plsvo_ctx_impl* c = CTX(ctx);
  if (in->n_features < 0 || in->n_ref_images <= 0 || in->n_cur_images <= 0 || in->cam.width <= 0 || in->cam.height <= 0 ||
      in->n_iter < 0 || in->n_pyr_levels < 1 || in->n_pyr_levels > PLSVO_MAX_LEVELS)
    return fail(c, PLSVO_ERR_INVALID, "match batch description");
  if (in->n_features == 0) return PLSVO_OK;
  if (!in->T_ref_w || !in->T_cur_w || !in->ref_index || !in->cur_index || !in->ref_px || !in->ref_f || !in->ref_level || !in->pos ||
      !in->px_cur || !out->px_cur || !out->success)
    return fail(c, PLSVO_ERR_INVALID, "match arrays missing");
  if (in->is_edgelet && !in->ref_grad) return fail(c, PLSVO_ERR_INVALID, "edgelets need ref_grad");
  const size_t n = (size_t)in->n_features;
  for (int l = 0; l < in->n_pyr_levels; ++l)
    if (!in->cur_img[l]) return fail(c, PLSVO_ERR_INVALID, "current pyramid level missing below n_pyr_levels");
  for (size_t i = 0; i < n; ++i) {
    const int l = in->ref_level[i];
    if (l < 0 || l >= PLSVO_MAX_LEVELS || !in->ref_img[l] || in->ref_index[i] < 0 || in->ref_index[i] >= in->n_ref_images ||
        in->cur_index[i] < 0 || in->cur_index[i] >= in->n_cur_images)
      return fail(c, PLSVO_ERR_INVALID, "match candidate refers to a missing level or frame");
  }
  CK(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  MatchArgs a;
  memset(&a, 0, sizeof a);
  a.n = in->n_features, a.n_iter = in->n_iter, a.n_pyr_levels = in->n_pyr_levels;
  a.width = in->cam.width, a.height = in->cam.height;
  a.fx = in->cam.fx, a.fy = in->cam.fy, a.cx = in->cam.cx, a.cy = in->cam.cy;
  int rc = stage_pyramid(c, c->m_ref_img, in->ref_img, in->ref_pitch, in->ref_stride, in->n_ref_images, a.width, a.height, s, a.ref_img,
                         a.ref_pitch, a.ref_stride);
  if (rc != PLSVO_OK) return rc;
  rc = stage_pyramid(c, c->m_cur_img, in->cur_img, in->cur_pitch, in->cur_stride, in->n_cur_images, a.width, a.height, s, a.cur_img,
                     a.cur_pitch, a.cur_stride);
  if (rc != PLSVO_OK) return rc;
  CK(up(c->m_T_ref, in->T_ref_w, (size_t)in->n_ref_images * 7, s, &a.T_ref_w));
  CK(up(c->m_T_cur, in->T_cur_w, (size_t)in->n_cur_images * 7, s, &a.T_cur_w));
  CK(up(c->m_ridx, in->ref_index, n, s, &a.ref_index));
  CK(up(c->m_cidx, in->cur_index, n, s, &a.cur_index));
  CK(up(c->m_px, in->ref_px, n * 2, s, &a.ref_px));
  CK(up(c->m_f, in->ref_f, n * 3, s, &a.ref_f));
  CK(up(c->m_lvl, in->ref_level, n, s, &a.ref_level));
  CK(up(c->m_edge, in->is_edgelet, n, s, &a.is_edgelet));
  CK(up(c->m_grad, in->is_edgelet ? in->ref_grad : nullptr, n * 2, s, &a.ref_grad));
  CK(up(c->m_pos, in->pos, n * 3, s, &a.pos));
  CK(up(c->m_pxc, in->px_cur, n * 2, s, &a.px_cur));
  CK(ensure(c->m_opx, n * 2 * sizeof(double)));
  CK(ensure(c->m_osucc, n));
  CK(ensure(c->m_olvl, n * sizeof(int32_t)));
  a.out_px = static_cast<double*>(c->m_opx.p);
  a.out_success = static_cast<uint8_t*>(c->m_osucc.p);
  a.out_level = static_cast<int32_t*>(c->m_olvl.p);
  if (out->A_cur_ref) {
    CK(ensure(c->m_oA, n * 4 * sizeof(double)));
    a.out_A = static_cast<double*>(c->m_oA.p);
    // rows the kernel leaves untouched (in-frame test failed) must come back as the caller passed them
    CK(cudaMemcpyAsync(a.out_A, out->A_cur_ref, n * 4 * sizeof(double), cudaMemcpyHostToDevice, s));
  }
  CK(kernel_timer(c, 0, s));
  CK(match_direct_kernel_launch(a, s));
  CK(kernel_timer(c, 1, s));
  c->launches += 1;
  CK(cudaMemcpyAsync(out->px_cur, a.out_px, n * 2 * sizeof(double), cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(out->success, a.out_success, n, cudaMemcpyDeviceToHost, s));
  if (out->search_level) CK(cudaMemcpyAsync(out->search_level, a.out_level, n * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  if (out->A_cur_ref) CK(cudaMemcpyAsync(out->A_cur_ref, a.out_A, n * 4 * sizeof(double), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  return PLSVO_OK;
}

static int structopt_batch_run_body(plsvo_ctx* ctx, const plsvo_structopt_batch* in, const plsvo_structopt_result* out) {
  plsvo_ctx_impl* c = CTX(ctx);
  if (in->n_points < 0 || in->n_segs < 0 || in->n_frames <= 0 || in->n_iter_pts < 0 || in->n_iter_segs < 0 || !in->T_f_w)
    return fail(c, PLSVO_ERR_INVALID, "structopt batch description");
  if (in->n_points + in->n_segs == 0) return PLSVO_OK;
  if (in->n_points > 0 && (!in->pt_obs_begin || !in->pt_pos || !out->pt_pos)) return fail(c, PLSVO_ERR_INVALID, "structopt point arrays missing");
  if (in->n_segs > 0 && (!in->seg_obs_begin || !in->seg_spos || !in->seg_epos || !out->seg_spos || !out->seg_epos))
    return fail(c, PLSVO_ERR_INVALID, "structopt segment arrays missing");
  const size_t np = (size_t)in->n_points, ns = (size_t)in->n_segs;
  const size_t npo = np ? (size_t)in->pt_obs_begin[np] : 0, nso = ns ? (size_t)in->seg_obs_begin[ns] : 0;
  // observation lists: monotone offsets, frame indices in range
  for (size_t i = 0; i < np; ++i)
    if (in->pt_obs_begin[i] > in->pt_obs_begin[i + 1] || in->pt_obs_begin[i] < 0) return fail(c, PLSVO_ERR_INVALID, "pt_obs_begin not monotone");
  for (size_t i = 0; i < ns; ++i)
    if (in->seg_obs_begin[i] > in->seg_obs_begin[i + 1] || in->seg_obs_begin[i] < 0) return fail(c, PLSVO_ERR_INVALID, "seg_obs_begin not monotone");
  if ((npo && (!in->pt_obs_frame || !in->pt_obs_f)) || (nso && (!in->seg_obs_frame || !in->seg_obs_sf || !in->seg_obs_ef)))
    return fail(c, PLSVO_ERR_INVALID, "structopt observation arrays missing");
  for (size_t o = 0; o < npo; ++o)
    if (in->pt_obs_frame[o] < 0 || in->pt_obs_frame[o] >= in->n_frames) return fail(c, PLSVO_ERR_INVALID, "observation refers to a missing frame");
  for (size_t o = 0; o < nso; ++o)
    if (in->seg_obs_frame[o] < 0 || in->seg_obs_frame[o] >= in->n_frames) return fail(c, PLSVO_ERR_INVALID, "observation refers to a missing frame");
  CK(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  StructOptArgs a;
  memset(&a, 0, sizeof a);
  a.n_points = in->n_points, a.n_segs = in->n_segs, a.n_iter_pts = in->n_iter_pts, a.n_iter_segs = in->n_iter_segs;
  CK(up(c->s_T, in->T_f_w, (size_t)in->n_frames * 7, s, &a.T_f_w));
  CK(up(c->s_pb, in->pt_obs_begin, np ? np + 1 : 0, s, &a.pt_obs_begin));
  CK(up(c->s_pf, in->pt_obs_frame, npo, s, &a.pt_obs_frame));
  CK(up(c->s_pof, in->pt_obs_f, npo * 3, s, &a.pt_obs_f));
  CK(up(c->s_pp, in->pt_pos, np * 3, s, &a.pt_pos));
  CK(up(c->s_sb, in->seg_obs_begin, ns ? ns + 1 : 0, s, &a.seg_obs_begin));
  CK(up(c->s_sf, in->seg_obs_frame, nso, s, &a.seg_obs_frame));
  CK(up(c->s_ssf, in->seg_obs_sf, nso * 3, s, &a.seg_obs_sf));
  CK(up(c->s_sef, in->seg_obs_ef, nso * 3, s, &a.seg_obs_ef));
  CK(up(c->s_sp, in->seg_spos, ns * 3, s, &a.seg_spos));
  CK(up(c->s_ep, in->seg_epos, ns * 3, s, &a.seg_epos));
  CK(ensure(c->s_out, (np * 3 + ns * 6) * sizeof(double) + (np + ns) * sizeof(int32_t) + 64));
  a.out_pt_pos = static_cast<double*>(c->s_out.p);
  a.out_seg_spos = a.out_pt_pos + np * 3;
  a.out_seg_epos = a.out_seg_spos + ns * 3;
  a.out_pt_iters = reinterpret_cast<int32_t*>(a.out_seg_epos + ns * 3);
  a.out_seg_iters = a.out_pt_iters + np;
  CK(kernel_timer(c, 0, s));
  CK(structopt_kernel_launch(a, s));
  CK(kernel_timer(c, 1, s));
  c->launches += 1;
  if (np) CK(cudaMemcpyAsync(out->pt_pos, a.out_pt_pos, np * 3 * sizeof(double), cudaMemcpyDeviceToHost, s));
  if (ns) {
    CK(cudaMemcpyAsync(out->seg_spos, a.out_seg_spos, ns * 3 * sizeof(double), cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(out->seg_epos, a.out_seg_epos, ns * 3 * sizeof(double), cudaMemcpyDeviceToHost, s));
  }
  if (np && out->pt_iters) CK(cudaMemcpyAsync(out->pt_iters, a.out_pt_iters, np * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  if (ns && out->seg_iters) CK(cudaMemcpyAsync(out->seg_iters, a.out_seg_iters, ns * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  return PLSVO_OK;
}

namespace {
// point seeds (lin == nullptr) and line seeds share staging; the line variant adds the end-point arrays
int seed_update_run(plsvo_ctx_impl* c, const plsvo_seed_batch* in, const plsvo_seed_result* out, const plsvo_line_seed_batch* lin,
                    const plsvo_line_seed_result* lout) {
  if (in->n_seeds < 0 || in->n_ref_images <= 0 || in->n_cur_images <= 0 || in->cam.width <= 0 || in->cam.height <= 0 ||
      in->n_iter < 0 || in->n_pyr_levels < 1 || in->n_pyr_levels > PLSVO_MAX_LEVELS || in->max_epi_search_steps < 0)
    return fail(c, PLSVO_ERR_INVALID, "seed batch description");
  if (in->n_seeds == 0) return PLSVO_OK;
  if (!in->T_ref_w || !in->T_cur_w || !in->ref_index || !in->cur_index || !in->ref_px || !in->ref_f || !in->ref_level || !in->a ||
      !in->b || !in->mu || !in->z_range || !in->sigma2 || !out->a || !out->b || !out->mu || !out->sigma2 || !out->status)
    return fail(c, PLSVO_ERR_INVALID, "seed arrays missing");
  if (!lin && in->is_edgelet && !in->ref_grad) return fail(c, PLSVO_ERR_INVALID, "edgelets need ref_grad");
  if (lin && (!lin->ref_sf || !lin->ref_ef || !lin->mu_e || !lin->z_range_e || !lin->sigma2_e || !lout->mu_e || !lout->sigma2_e))
    return fail(c, PLSVO_ERR_INVALID, "line-seed end-point arrays missing");
  const size_t n = (size_t)in->n_seeds;
  for (int l = 0; l < in->n_pyr_levels; ++l) {
    if (!in->cur_img[l]) return fail(c, PLSVO_ERR_INVALID, "current pyramid level missing below n_pyr_levels");
    // the reference strides the ZMSSD patch with Mat::cols (matcher.cpp:380-382): only dense images mean the same thing
    if (in->cur_pitch[l] != (size_t)(in->cam.width >> l)) return fail(c, PLSVO_ERR_INVALID, "current images must be dense (pitch == level width)");
  }
  for (size_t i = 0; i < n; ++i) {
    const int l = in->ref_level[i];
    if (l < 0 || l >= PLSVO_MAX_LEVELS || !in->ref_img[l] || in->ref_index[i] < 0 || in->ref_index[i] >= in->n_ref_images ||
        in->cur_index[i] < 0 || in->cur_index[i] >= in->n_cur_images)
      return fail(c, PLSVO_ERR_INVALID, "seed refers to a missing level or frame");
  }
  CK(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  SeedArgs a;
  memset(&a, 0, sizeof a);
  a.n = in->n_seeds, a.n_iter = in->n_iter, a.n_pyr_levels = in->n_pyr_levels, a.max_epi_search_steps = in->max_epi_search_steps;
  a.align_1d = in->align_1d, a.subpix_refinement = in->subpix_refinement, a.edgelet_filtering = in->epi_search_edgelet_filtering;
  a.edgelet_max_angle = in->epi_search_edgelet_max_angle, a.convergence_thresh = in->seed_convergence_sigma2_thresh;
  a.width = in->cam.width, a.height = in->cam.height;
  a.fx = in->cam.fx, a.fy = in->cam.fy, a.cx = in->cam.cx, a.cy = in->cam.cy;
  int rc = stage_pyramid(c, c->m_ref_img, in->ref_img, in->ref_pitch, in->ref_stride, in->n_ref_images, a.width, a.height, s, a.ref_img,
                         a.ref_pitch, a.ref_stride);
  if (rc != PLSVO_OK) return rc;
  rc = stage_pyramid(c, c->m_cur_img, in->cur_img, in->cur_pitch, in->cur_stride, in->n_cur_images, a.width, a.height, s, a.cur_img,
                     a.cur_pitch, a.cur_stride);
  if (rc != PLSVO_OK) return rc;
  CK(up(c->m_T_ref, in->T_ref_w, (size_t)in->n_ref_images * 7, s, &a.T_ref_w));
  CK(up(c->m_T_cur, in->T_cur_w, (size_t)in->n_cur_images * 7, s, &a.T_cur_w));
  CK(up(c->m_ridx, in->ref_index, n, s, &a.ref_index));
  CK(up(c->m_cidx, in->cur_index, n, s, &a.cur_index));
  CK(up(c->m_px, in->ref_px, n * 2, s, &a.ref_px));
  CK(up(c->m_f, in->ref_f, n * 3, s, &a.ref_f));
  CK(up(c->m_lvl, in->ref_level, n, s, &a.ref_level));
  CK(up(c->m_edge, lin ? nullptr : in->is_edgelet, n, s, &a.is_edgelet));
  CK(up(c->m_grad, (!lin && in->is_edgelet) ? in->ref_grad : nullptr, n * 2, s, &a.ref_grad));
  if (lin) {
    CK(up(c->m_pos, lin->ref_sf, n * 3, s, &a.ref_sf));
    CK(up(c->m_pxc, lin->ref_ef, n * 3, s, &a.ref_ef));
    CK(up(c->d_smu_e, lin->mu_e, n, s, &a.mu_e));
    CK(up(c->d_szr_e, lin->z_range_e, n, s, &a.z_range_e));
    CK(up(c->d_ssig_e, lin->sigma2_e, n, s, &a.sigma2_e));
  }
  CK(up(c->d_sa, in->a, n, s, &a.a));
  CK(up(c->d_sb, in->b, n, s, &a.b));
  CK(up(c->d_smu, in->mu, n, s, &a.mu));
  CK(up(c->d_szr, in->z_range, n, s, &a.z_range));
  CK(up(c->d_ssig, in->sigma2, n, s, &a.sigma2));
  // outputs: [px_cur_e 2n f64][px_cur 2n f64][depth n f64][depth_e n f64][a b mu sigma2 mu_e sigma2_e n f32 each][status n i32][converged n u8]
  CK(ensure(c->d_sout, n * (16 + 16 + 8 + 8 + 24 + 4 + 1) + 64));
  a.out_px_cur_e = static_cast<double*>(c->d_sout.p);
  a.out_px_cur = a.out_px_cur_e + 2 * n;
  a.out_depth = a.out_px_cur + 2 * n;
  a.out_depth_e = a.out_depth + n;
  a.out_a = reinterpret_cast<float*>(a.out_depth_e + n);
  a.out_b = a.out_a + n, a.out_mu = a.out_b + n, a.out_sigma2 = a.out_mu + n;
  a.out_mu_e = a.out_sigma2 + n, a.out_sigma2_e = a.out_mu_e + n;
  a.out_status = reinterpret_cast<int32_t*>(a.out_sigma2_e + n);
  a.out_converged = reinterpret_cast<uint8_t*>(a.out_status + n);
  CK(kernel_timer(c, 0, s));
  CK(lin ? line_seed_update_kernel_launch(a, s) : seed_update_kernel_launch(a, s));
  CK(kernel_timer(c, 1, s));
  c->launches += 1;
  CK(cudaMemcpyAsync(out->a, a.out_a, n * 4, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(out->b, a.out_b, n * 4, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(out->mu, a.out_mu, n * 4, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(out->sigma2, a.out_sigma2, n * 4, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(out->status, a.out_status, n * 4, cudaMemcpyDeviceToHost, s));
  if (out->converged) CK(cudaMemcpyAsync(out->converged, a.out_converged, n, cudaMemcpyDeviceToHost, s));
  if (out->depth) CK(cudaMemcpyAsync(out->depth, a.out_depth, n * 8, cudaMemcpyDeviceToHost, s));
  if (out->px_cur) CK(cudaMemcpyAsync(out->px_cur, a.out_px_cur, n * 16, cudaMemcpyDeviceToHost, s));
  if (lin) {
    CK(cudaMemcpyAsync(lout->mu_e, a.out_mu_e, n * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(lout->sigma2_e, a.out_sigma2_e, n * 4, cudaMemcpyDeviceToHost, s));
    if (lout->depth_e) CK(cudaMemcpyAsync(lout->depth_e, a.out_depth_e, n * 8, cudaMemcpyDeviceToHost, s));
    if (lout->px_cur_e) CK(cudaMemcpyAsync(lout->px_cur_e, a.out_px_cur_e, n * 16, cudaMemcpyDeviceToHost, s));
  }
  CK(cudaStreamSynchronize(s));
  return PLSVO_OK;
}
}  // namespace

extern "C" int plsvo_seed_update_batch_run(plsvo_ctx* ctx, const plsvo_seed_batch* in, const plsvo_seed_result* out) {
  if (!ctx || !in || !out) return PLSVO_ERR_INVALID;
  return settled(CTX(ctx), seed_update_run(CTX(ctx), in, out, nullptr, nullptr));
}

extern "C" int plsvo_line_seed_update_batch_run(plsvo_ctx* ctx, const plsvo_line_seed_batch* in, const plsvo_line_seed_result* out) {
  if (!ctx || !in || !out) return PLSVO_ERR_INVALID;
  return settled(CTX(ctx), seed_update_run(CTX(ctx), &in->seeds, &out->seeds, in, out));
}

// exported forms of the three bodies above (see settled())
extern "C" int plsvo_pyramid_batch_run(plsvo_ctx* ctx, const plsvo_pyramid_batch* in, const plsvo_pyramid_result* out) {
  if (!ctx || !in || !out) return PLSVO_ERR_INVALID;
  return settled(CTX(ctx), pyramid_batch_run_body(ctx, in, out));
}

extern "C" int plsvo_match_direct_batch_run(plsvo_ctx* ctx, const plsvo_match_batch* in, const plsvo_match_result* out) {
  if (!ctx || !in || !out) return PLSVO_ERR_INVALID;
  return settled(CTX(ctx), match_direct_batch_run_body(ctx, in, out));
}

extern "C" int plsvo_structopt_batch_run(plsvo_ctx* ctx, const plsvo_structopt_batch* in, const plsvo_structopt_result* out) {
  if (!ctx || !in || !out) return PLSVO_ERR_INVALID;
  return settled(CTX(ctx), structopt_batch_run_body(ctx, in, out));
}
