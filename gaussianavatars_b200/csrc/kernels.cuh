// Internal launcher declarations + small device helpers shared by the .cu files.
#pragma once
#include "common.cuh"

namespace gab {

// SH constants (values of utils/sh_utils.py:26-43)
#define SH_C0 0.28209479177387814f
#define SH_C1 0.4886025119029199f
#define SH_C2_0 1.0925484305920792f
#define SH_C2_1 -1.0925484305920792f
#define SH_C2_2 0.31539156525252005f
#define SH_C2_3 -1.0925484305920792f
#define SH_C2_4 0.5462742152960396f
#define SH_C3_0 -0.5900435899266435f
#define SH_C3_1 2.890611442640554f
#define SH_C3_2 -0.4570457994644658f
#define SH_C3_3 0.3731763325901154f
#define SH_C3_4 -0.4570457994644658f
#define SH_C3_5 1.445305721320277f
#define SH_C3_6 -0.5900435899266435f

void count_launch();
int tune_get(int knob);  // api.cu: current value of a gab200_tune() knob

// Exact per-tile-row span of the region where a splat can reach alpha >= 1/255:
//   q(d) = 1/2 (A dx^2 + C dy^2) + B dx dy <= ln(255 * opacity)          (the blend's own accept test)
// For tile row ty the pixel centres have dy in [16 ty - py, 16 ty + 15 - py]; the x-extent of the ellipse over
// that band is closed-form (extreme point if it lies in the band, else the better band edge).  The span is
// intersected with the reference's 3-sigma bounding-square columns [rx0, rx1) so the emitted instance list is
// always a SUBSEQUENCE of the reference's.  Margins: +0.01 in the exponent (alpha down to 0.99/255 kept) and
// +-0.02 px, i.e. only pairs that contribute exactly nothing are dropped.
struct TileSpan {
  bool any, full;
  float px, py, A, B, tau2A, det, dxmax, ystar, ymax;
  int rx0, rx1;
  __device__ __forceinline__ TileSpan(float px_, float py_, float A_, float B_, float C_, float opacity, int rx0_,
                                      int rx1_)
      : px(px_), py(py_), A(A_), B(B_), rx0(rx0_), rx1(rx1_) {
    const float tau = logf(255.f * opacity) + 0.01f;
    det = A_ * C_ - B_ * B_;
    const bool pd = (det > 0.f) && (A_ > 0.f) && (C_ > 0.f) && (det < 3.0e38f);
    any = tau > 0.f;
    full = !pd || !(tau < 3.0e38f);
    const float tau2 = 2.f * tau;
    tau2A = tau2 * A_;
    dxmax = sqrtf(fmaxf(0.f, tau2 * C_ / det));
    ymax = sqrtf(fmaxf(0.f, tau2 * A_ / det));
    ystar = (B_ / C_) * dxmax;
  }
  __device__ __forceinline__ float half_width(float dy) const { return sqrtf(fmaxf(0.f, tau2A - det * dy * dy)); }
  __device__ __forceinline__ void row(int ty, int& cx0, int& cx1) const {
    if (!any) { cx0 = cx1 = rx0; return; }
    if (full) { cx0 = rx0; cx1 = rx1; return; }
    const float a = (float)(ty * GAB_TILE) - py, b = a + (float)(GAB_TILE - 1);
    const float lo = fmaxf(a, -ymax) - 0.02f, hi = fminf(b, ymax) + 0.02f;
    if (lo > hi) { cx0 = cx1 = rx0; return; }
    float xr, xl;
    const float hl = half_width(lo), hh = half_width(hi);
    if (-ystar >= lo && -ystar <= hi) xr = dxmax;
    else xr = fmaxf((-B * lo + hl) / A, (-B * hi + hh) / A);
    if (ystar >= lo && ystar <= hi) xl = -dxmax;
    else xl = fminf((-B * lo - hl) / A, (-B * hi - hh) / A);
    const float X0 = px + xl - 0.02f, X1 = px + xr + 0.02f;
    int t0 = (int)ceilf((X0 - (float)(GAB_TILE - 1)) * (1.0f / GAB_TILE));
    int t1 = (int)floorf(X1 * (1.0f / GAB_TILE)) + 1;
    cx0 = min(max(t0, rx0), rx1);
    cx1 = max(min(t1, rx1), cx0);
  }
};

// ---- launchers (each counts its launches) ----
// Per-splat depth sort as a bucket sort (binning.cu header): bookkeeping arrays in the geometry buffer.
#define GAB_DEPTH_BUCKET_CAP 2048   // splats one bucket may hold before the frame falls back to the radix path
// the frame counters of the public header (GAB200_CTR_*) + two private words: the 64-bit instance total
// (meta[GAB_META_TOTAL64 .. +1], 8-byte aligned), from which GAB200_CTR_NUM_RENDERED_HI is published
#define GAB_DEPTH_META_WORDS (GAB200_NUM_COUNTERS + 2)
#define GAB_META_TOTAL64 GAB200_NUM_COUNTERS
struct DepthBuckets {
  uint32_t* counts;     // [nb] splats per bucket           } zeroed together with meta before preprocess
  uint32_t* tiles;      // [nb] instances per bucket        }
  uint32_t* meta;       // [GAB_DEPTH_META_WORDS]           }
  uint32_t* start;      // [nb] exclusive prefix of counts
  uint32_t* tile_base;  // [nb] exclusive prefix of tiles
  uint32_t* rank;       // [P]  arrival rank of the splat inside its bucket
  uint32_t nb;          // buckets (power of two)
  uint32_t lo, hi;      // hinted key range; keys outside are clamped to the end buckets (order is preserved)
  float scale;          // nb / (hi - lo + 1)
  int enabled;          // 0: only meta[0..1] (min/max key) are maintained
};
// Monotonic non-decreasing in `key` (u32->f32 conversion, multiply by a positive constant and truncation all are),
// which is all the bucket sort needs.  Evaluated in preprocess.cu only (one translation unit, one set of flags).
__device__ __forceinline__ uint32_t depth_bucket(uint32_t key, const DepthBuckets& d) {
  if (key <= d.lo) return 0u;
  if (key >= d.hi) return d.nb - 1u;
  const uint32_t b = (uint32_t)(__uint2float_rz(key - d.lo) * d.scale);
  return b < d.nb ? b : d.nb - 1u;
}
// tile_count != nullptr: also count the instances of every tile (counting tile sort, tile_sort.cu)
void launch_preprocess(const gab200_forward_args& a, SplatRec* rec, SplatAux* aux, uint32_t* tiles_touched,
                       uint8_t* clamped, uint32_t* depth_keys, uint32_t* ids, const DepthBuckets& buckets,
                       uint32_t* tile_count, cudaStream_t stream);
// depth_keys [P] (by splat) -> sorted_ids [M] in (key, id) order and offsets [M] = inclusive instance counts
// also publishes the frame counters (capacity, seq, overflow) of the bucket-sorted frame
void launch_depth_bucket_sort(int P, const DepthBuckets& buckets, const uint32_t* depth_keys,
                              const uint32_t* tiles_touched, uint32_t* scratch_keys, uint32_t* sorted_ids,
                              uint32_t* offsets, uint32_t capacity, uint32_t seq, uint32_t* sticky_overflow,
                              cudaStream_t stream);
void launch_bind_activate(const gab200_forward_args& a, float* means3D, float* opacities, float* scales, float* cov3D,
                          cudaStream_t stream);
void launch_mark_visible(int P, const float* means3D, const float* V, uint8_t* present, cudaStream_t stream);
// counters[NUM_LISTED] (+ NUM_RENDERED from offsets when given) of a radix-sorted frame (P > 0; pass 0 for a
// bucket-sorted one, whose kernels wrote them), capacity and sequence number
void launch_publish_counters(uint32_t* counters, const uint32_t* offsets, int P, uint32_t capacity, uint32_t seq,
                             uint32_t* sticky_overflow, cudaStream_t stream);
// `capacity`: instances the key/value arrays hold -- anything beyond is dropped (the frame's counters say so);
// counters[BUCKET_OVERFLOW] != 0 (depth order unusable) emits nothing.
void launch_emit_keys(int P, int gx, int gy, const SplatRec* rec, const SplatAux* aux, const uint32_t* order,
                      const uint32_t* offsets, const uint32_t* order_count, const uint32_t* counters, uint32_t capacity,
                      uint32_t* cursor, uint32_t* keys, uint32_t* vals, int exact_binning, cudaStream_t stream);
// keys[0..N) sorted; entries with key >= tiles are padding (sentinel) behind the last real instance
void launch_tile_ranges(int64_t N, uint32_t tiles, const uint32_t* keys, uint2* ranges, cudaStream_t stream);
void launch_expand_keys(int64_t N, const uint32_t* tile_keys, const uint32_t* ids, const SplatAux* aux, uint64_t* out,
                        cudaStream_t stream);
// tile_sort.cu
#define GAB_TILE_SORT_SMEM 2048  // entries one CTA sorts in shared memory; longer tile lists take the bitmap kernel
// tile_count != nullptr: ranges / cursors / counters[NUM_RENDERED] from the per-tile counts (ranges cut at `clamp`);
// always: heaviest-first tile order + heavy/light split points (order_info[0..1]) + number of long tiles ([2])
void launch_tile_scan_order(int tiles, const uint32_t* tile_count, uint32_t clamp, uint2* ranges, uint32_t* cursor,
                            uint32_t* order, uint32_t* order_info, uint32_t* counters, int heavy_fwd, int heavy_bwd,
                            cudaStream_t stream);
// every tile's (rank, id) segment sorted by rank; ids written back in place
void launch_tile_sort(int tiles, const uint2* ranges, const uint32_t* order, const uint32_t* order_info, uint32_t* keys,
                      uint32_t* vals, const uint32_t* rank_to_id, const uint32_t* listed, int P, cudaStream_t stream);
void launch_expand_keys_by_range(int tiles, const uint2* ranges, const uint32_t* ids, const SplatAux* aux, uint64_t* out,
                                 cudaStream_t stream);

// binning.cu (cub)
size_t scan_temp_bytes(int P);
cudaError_t run_scan(void* temp, size_t temp_bytes, const uint32_t* order, const uint32_t* tiles_touched, uint32_t* out,
                     int P, cudaStream_t stream);
size_t sort_temp_bytes(int64_t N, int end_bit);
cudaError_t run_sort(void* temp, size_t temp_bytes, uint32_t* keys_a, uint32_t* keys_b, uint32_t* vals_a,
                     uint32_t* vals_b, int64_t N, int end_bit, int* selector_out, cudaStream_t stream);

// blend.cu
void launch_blend_forward(int W, int H, const uint2* ranges, const uint32_t* order, const uint32_t* order_info,
                          const uint32_t* point_list, const SplatRec* rec,
                          const float* bg, float* out_color, float* final_T, uint32_t* n_contrib, uint8_t* strip_mask,
                          cudaStream_t stream);
void launch_blend_backward(int W, int H, const uint2* ranges, const uint32_t* order, const uint32_t* order_info,
                           const uint32_t* point_list, const SplatRec* rec,
                           const float* bg, const float* final_T, const uint32_t* n_contrib, const float* dL_dpix,
                           const uint8_t* strip_mask, float* g2d, cudaStream_t stream);

// preprocess_bwd.cu
void launch_preprocess_backward(const gab200_backward_args& b, const SplatRec* rec, const SplatAux* aux,
                                const uint8_t* clamped, const float* g2d, float* face_scratch, cudaStream_t stream);
#define GAB_FACE_GRAD_STRIDE 13  // per-splat face-frame gradient record: centre 3, orientation 9, scale 1

// face_frame.cu
void launch_face_frame_forward(int F, const float* verts, const int32_t* faces, float* fc, float* fR, float* fs,
                               cudaStream_t stream);
void launch_face_frame_backward(int F, const float* verts, const int32_t* faces, const float* g_fc, const float* g_fR,
                                const float* g_fs, float* g_verts, cudaStream_t stream);

// flame.cu
size_t flame_workspace_bytes(int V, int NB);
void launch_flame_forward(const gab200_flame_args& a, cudaStream_t stream);
void launch_flame_backward(const gab200_flame_args& a, const float* g_verts, cudaStream_t stream);

// loss.cu
void launch_l1_loss_u8(int64_t n, const float* img, const uint8_t* gt, const float* upstream, float* grad, float* loss,
                       cudaStream_t stream);

void launch_photometric_loss(int C, int H, int W, const float* img, const void* gt, int gt_is_u8, float lambda,
                             float* grad, float* loss, float* scratch, cudaStream_t stream);

// densify.cu
size_t densify_scratch_bytes(int P, int F);
cudaError_t launch_densify_plan(const gab200_densify_args& a, cudaStream_t stream);
cudaError_t launch_densify_apply(const gab200_densify_args& a, const gab200_densify_out& o, cudaStream_t stream);

// regularize.cu
cudaError_t launch_regularize_forward(const gab200_regularize_args& a, cudaStream_t stream);
cudaError_t launch_regularize_backward(const gab200_regularize_args& a, const float* g_out, cudaStream_t stream);

// nvls.cu
void launch_nvls_allreduce(float* mc, int64_t n, int rank, int world, cudaStream_t stream);

// optim.cu
void launch_adam(int num_segments, const gab200_adam_segment* segs, int64_t step, double beta1, double beta2, double eps,
                 cudaStream_t stream);

}  // namespace gab
