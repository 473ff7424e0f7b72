/*
 * gab200_rasterizer.h -- C ABI of the B200-native differentiable Gaussian-splat rasterizer with fused
 * FLAME mesh binding (libgaussianavatars_b200.so).
 *
 * This is the drop-in boundary for the one native operator GaussianAvatars calls on its hot path:
 *   reference call site ........ gaussian_renderer/__init__.py:15,37-52,86-94
 *   reference native module .... diff_gaussian_rasterization._C (submodule graphdeco-inria/diff-gaussian-rasterization
 *                                @59f5f77, ABSENT from /root/reference; its pybind surface is
 *                                rasterize_gaussians / rasterize_gaussians_backward / mark_visible, SURVEY.md 2.2, 8a/a8-a9)
 * Each entry point below names the reference interface it replaces.
 *
 * Conventions
 *   - Every pointer is a DEVICE pointer owned by the caller unless stated otherwise; fp32 unless stated.
 *   - Matrices are the row-major flatten of the (4,4) tensors GaussianAvatars builds
 *     (world_view_transform = W2C^T, full_proj_transform = (P W2C)^T; scene/cameras.py:44-46).
 *   - Nothing a call leaves behind in the library affects a later result: what persists is a launch counter,
 *     the opt-in stage/host timers (atomics), the tuning knobs of gab200_tune(), and per host thread a 64-byte
 *     pinned read-back slot (hints such as binning_hint / depth_hint_* travel through the caller; the layout of
 *     the three scratch buffers is a pure function of the arguments).  Thread-safe per stream; no
 *     exceptions cross the ABI: functions return >= 0 on success and a negative gab200_status on failure
 *     (gab200_status_string() explains it).
 *   - Scratch memory is obtained through caller-supplied allocation callbacks, mirroring the reference
 *     module's three resizable byte buffers (geometry / binning / image; SURVEY.md 8a/a9).  The callbacks
 *     are invoked on the calling host thread, must return device memory aligned to 256 B that stays valid
 *     until the matching gab200_backward() has run (or is never called).
 */
#ifndef GAB200_RASTERIZER_H
#define GAB200_RASTERIZER_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GAB200_ABI_VERSION 3

typedef enum gab200_status {
  GAB200_OK = 0,
  GAB200_ERR_INVALID_ARGUMENT = -1, /* bad shape / missing pointer / inconsistent option        */
  GAB200_ERR_CUDA = -2,             /* a CUDA runtime call or kernel failed (see cudaGetLastError) */
  GAB200_ERR_ALLOC = -3,            /* an allocation callback returned NULL                       */
  GAB200_ERR_ARCH = -4,             /* device is not sm_100 class                                 */
  GAB200_ERR_OVERFLOW = -5          /* more than 2^32-1 (splat,tile) instances                    */
} gab200_status;

/* Input interpretation. */
typedef enum gab200_input_mode {
  /* Reference surface: means3D world-space, scales already exp()-activated, rotations unit wxyz (used as given),
   * opacities already sigmoid()-activated -- exactly what render() passes today
   * (gaussian_renderer/__init__.py:54-94 <- scene/gaussian_model.py:113-160). */
  GAB200_INPUT_ACTIVATED = 0,
  /* Fused surface: the RAW parameters of GaussianModel (_xyz local, _scaling log, _rotation unnormalised,
   * _opacity logit, _features_dc/_features_rest) plus the per-face frame; the binding transform of
   * scene/gaussian_model.py:113-160 runs inside the preprocess kernel.  binding == NULL means identity frame. */
  GAB200_INPUT_BOUND_RAW = 1
} gab200_input_mode;

/* How gab200_forward learns N, the number of (splat,tile) instances of the frame (the reference copies it to the
 * host in the middle of every forward to size its binning buffer: rasterizer_impl.cu, SURVEY.md 2.4 K2 / 7.3). */
typedef enum gab200_sync_mode {
  /* One host wait in the MIDDLE of the forward (after preprocess + per-splat depth sort): the binning buffer is
   * sized for exactly N.  Needs no hint; this is what the first frame of a model uses. */
  GAB200_SYNC_EXACT = 0,
  /* binning_hint (> 0) is a hard CAPACITY: the whole forward is enqueued without waiting, then the host waits for
   * the frame counters at the END of the call (they were written long before in the common case) and, only if the
   * frame needed more than the capacity or the depth-bucket hint did not fit, re-enqueues the affected stages with
   * the exact size.  The result is the same as GAB200_SYNC_EXACT's, bit for bit; the GPU never idles behind the host. */
  GAB200_SYNC_LATE = 1,
  /* Never waits (required while the stream is being captured into a CUDA graph).  The frame counters are copied
   * to `counters_host`; the caller inspects them whenever it likes (gab200_counters_ok()).  A frame that overflowed
   * its capacity was rendered from a truncated instance list (memory-safe, wrong image): redo it with a larger
   * binning_hint. */
  GAB200_SYNC_NONE = 2
} gab200_sync_mode;

/* Frame counters (device: gab200_frame_state.device_counters; host copy: counters_host), 8 x uint32. */
enum {
  GAB200_CTR_NOT_MIN_DEPTH_KEY = 0, /* ~(smallest depth key among the splats that emitted instances) */
  GAB200_CTR_MAX_DEPTH_KEY = 1,
  GAB200_CTR_NUM_RENDERED = 2,      /* N the frame needs (may exceed the capacity it was given) */
  GAB200_CTR_NUM_LISTED = 3,        /* splats with at least one instance */
  GAB200_CTR_BUCKET_OVERFLOW = 4,   /* != 0: a depth bucket outgrew shared memory (depth_hint_* did not fit this frame) */
  GAB200_CTR_CAPACITY = 5,          /* capacity the binning stages ran with */
  GAB200_CTR_SEQ = 6,               /* caller's frame_seq echoed back: tells a finished copy from a stale one */
  GAB200_CTR_NUM_RENDERED_HI = 7,   /* bits 32.. of the instance total: non-zero = more than 2^32 - 1 instances (the 32-bit
                                       offsets wrapped: GAB200_ERR_OVERFLOW) */
  GAB200_NUM_COUNTERS = 8
};

typedef void* (*gab200_alloc_fn)(void* user, size_t bytes);

/* Everything one frame's forward needs.  Replaces the argument list of
 * diff_gaussian_rasterization._C.rasterize_gaussians (SURVEY.md 3.3 / Appendix B.6). */
typedef struct gab200_forward_args {
  uint32_t abi_version;    /* = GAB200_ABI_VERSION */
  int32_t input_mode;      /* gab200_input_mode */
  int32_t P;               /* number of splats */
  int32_t sh_degree;       /* active SH degree D (0..3) */
  int32_t sh_coeffs;       /* M: coefficients stored per splat (1,4,9,16); 0 with colors_precomp */
  int32_t image_width, image_height;
  float tanfovx, tanfovy, scale_modifier;
  int32_t prefiltered;     /* accepted for signature parity; the near-plane cull is always applied */
  int32_t debug;           /* 1: synchronise + check after every stage (reference `debug=` flag) */
  int32_t need_backward;   /* 0: inference -- per-pixel state for backward is not written */
  int32_t binning_hint;    /* expected number of (splat,tile) instances (0 = unknown), e.g. last frame's N * 1.25.
                              GAB200_SYNC_EXACT: the binning buffer is requested BEFORE the host sync that reads N back
                              (allocation off the critical path; requested again only if N exceeds the hint).
                              GAB200_SYNC_LATE / NONE: the capacity the binning stages run with (see gab200_sync_mode) */
  int32_t exact_binning;   /* 1: emit the reference's full 3-sigma bounding-square instance list;
                              0: additionally drop (splat,tile) pairs that provably contribute nothing
                                 (alpha < 1/255 over the whole tile): image/gradients unchanged */
  uint32_t depth_hint_lo;  /* expected range of the visible splats' depth keys (fp32 bit patterns of view-space z), e.g.
                              the previous frame's gab200_frame_state.depth_key_min/max widened a little; hi <= lo = unknown.
                              With a hint the per-splat depth sort runs as a bucket sort (3 small launches) instead of
                              cub::DeviceRadixSort + DeviceScan (8 launches); the result is the same bit for bit, and a
                              hint that turns out wrong only costs the time of the radix path on top. */
  uint32_t depth_hint_hi;
  int32_t sync_mode;       /* gab200_sync_mode */
  uint32_t frame_seq;      /* any value; echoed in counters[GAB200_CTR_SEQ] */
  uint32_t* counters_host; /* HOST pointer (pinned memory), GAB200_NUM_COUNTERS words, or NULL: where the frame counters
                              are copied.  Required for GAB200_SYNC_NONE; the other modes fall back to a slot the
                              library keeps per host thread. */
  uint32_t* overflow_flag; /* DEVICE pointer or NULL: the library ORs 1 into it when the frame needed more than its
                              capacity or its depth buckets overflowed, and never clears it -- a replayed CUDA graph
                              (GAB200_SYNC_NONE) cannot lose an overflow between two looks at the counters */

  /* camera block */
  const float* bg;         /* [3] */
  const float* viewmatrix; /* [16] */
  const float* projmatrix; /* [16] */
  const float* campos;     /* [3] */

  /* splat attributes (meaning depends on input_mode) */
  const float* means3D;        /* [P,3]  world xyz | raw _xyz (face-local) */
  const float* opacities;      /* [P]    sigmoid-ed | raw logit */
  const float* scales;         /* [P,3]  exp-ed | raw log;            NULL iff cov3D_precomp */
  const float* rotations;      /* [P,4]  wxyz unit | raw unnormalised; NULL iff cov3D_precomp */
  const float* cov3D_precomp;  /* [P,6]  xx,xy,xz,yy,yz,zz; ACTIVATED mode only, else NULL */
  const float* shs;            /* [P,M,3] ACTIVATED mode: concatenated SH; NULL with colors_precomp */
  const float* sh_dc;          /* [P,1,3]   BOUND_RAW mode: _features_dc   (no torch.cat needed) */
  const float* sh_rest;        /* [P,M-1,3] BOUND_RAW mode: _features_rest (may be NULL when M==1) */
  const float* colors_precomp; /* [P,3]  overrides SH when non-NULL */

  /* mesh binding (BOUND_RAW mode; scene/flame_gaussian_model.py:137-147) */
  const int32_t* binding;        /* [P] face index per splat, or NULL (identity frame) */
  int32_t num_faces;             /* F */
  const float* face_center;      /* [F,3] */
  const float* face_orien_mat;   /* [F,3,3] row-major, columns a0 a1 a2 */
  const float* face_scaling;     /* [F] */

  /* outputs */
  float* out_color;   /* [3,H,W] */
  int32_t* radii;     /* [P] */
  uint8_t* visibility; /* [P] or NULL: radii > 0 as bytes -- render()'s `visibility_filter`
                          (gaussian_renderer/__init__.py:100) without a separate compare kernel */

  /* scratch (the reference's geomBuffer / binningBuffer / imgBuffer) */
  gab200_alloc_fn alloc_geom, alloc_binning, alloc_image;
  void* alloc_user;
} gab200_forward_args;

/* Host-side handle to the state a forward leaves behind for its backward (what the reference keeps as
 * num_rendered + the three byte buffers in the autograd ctx). Plain data; copy freely. */
typedef struct gab200_frame_state {
  int64_t num_rendered;       /* N: (splat,tile) instances sorted and blended */
  int64_t num_candidates;     /* instances of the reference's bounding-square list (== N when exact_binning) */
  void* geom_buffer;
  void* binning_buffer;
  void* image_buffer;
  size_t geom_bytes, binning_bytes, image_bytes;
  int32_t sorted_selector;    /* which half of the sort double-buffer holds the sorted stream */
  int32_t sort_bits;          /* key width of the per-instance (stage B) radix sort: bits(tile id) */
  int32_t depth_bits;         /* key width of the per-splat (stage A) radix sort: 32 (the fp32 depth pattern); the two
                                 stable stages together are the reference's LSD sort of (tile << 32 | depth) */
  uint32_t depth_prefix;      /* reserved (0) */
  int64_t binning_capacity;   /* instances the binning buffer was carved for (>= num_rendered; = binning_hint when the
                                 speculative allocation was large enough) */
  uint32_t depth_key_min;     /* smallest / largest depth key among the splats that emitted instances (min > max: none) */
  uint32_t depth_key_max;
  int32_t depth_sort_path;    /* 0: radix sort (no hint); 1: bucket sort; 2: bucket sort overflowed, radix sort redone */
  int32_t attempts;           /* 1 + number of times stages were re-enqueued (GAB200_SYNC_LATE only; else 1) */
  int32_t tile_sort_path;     /* 0: cub::DeviceRadixSort over the instances; 1: counting sort by tile + per-tile rank sort */
  int32_t reserved0;
  const uint32_t* device_counters; /* GAB200_NUM_COUNTERS words inside the geometry buffer (valid as long as it is) */
} gab200_frame_state;

/* Forward.  Returns num_rendered (>= 0) or a negative gab200_status.  With GAB200_SYNC_NONE the count is not known
 * when the call returns: it returns 0 and sets state_out->num_rendered = -1.  Enqueues on `stream` (cudaStream_t as
 * void*).  Host<->device synchronisation: see gab200_sync_mode. */
int64_t gab200_forward(const gab200_forward_args* args, gab200_frame_state* state_out, void* stream);

/* 1 if a GAB200_SYNC_NONE frame whose counters are in `counters` (HOST copy) was rendered from its complete instance
 * list, 0 if it overflowed (capacity or depth buckets) and has to be redone, -1 if the copy has not landed yet
 * (counters[GAB200_CTR_SEQ] != frame_seq). */
int32_t gab200_counters_ok(const uint32_t* counters, uint32_t frame_seq);

/* Gradients.  Replaces rasterize_gaussians_backward (SURVEY.md 3.4).  All outputs are written in full
 * (zeros where a splat received no gradient); NULL outputs are skipped where noted.
 * ACTIVATED mode: dL_dmeans3D [P,3], dL_dmeans2D [P,3] (x,y in NDC units, z = 0), dL_dopacity [P],
 *   dL_dcolors [P,3] (also the colors_precomp gradient), dL_dshs [P,M,3] | NULL, dL_dscales [P,3] | NULL,
 *   dL_drotations [P,4] | NULL, dL_dcov3D [P,6].
 * BOUND_RAW mode: same pointers are gradients w.r.t. the RAW parameters (_xyz, logit, log-scale, raw quaternion);
 *   dL_dsh_dc [P,1,3], dL_dsh_rest [P,M-1,3]; plus the face-frame gradients dL_dface_center [F,3],
 *   dL_dface_orien_mat [F,3,3], dL_dface_scaling [F] (accumulated; caller zero-initialises NOTHING -- the library does).
 */
typedef struct gab200_backward_args {
  uint32_t abi_version;
  const gab200_forward_args* fwd;   /* the same inputs the forward saw */
  const gab200_frame_state* state;
  const float* dL_dout_color;       /* [3,H,W] */
  float* dL_dmeans3D;
  float* dL_dmeans2D;
  float* dL_dopacity;
  float* dL_dcolors;
  float* dL_dshs;
  float* dL_dsh_dc;
  float* dL_dsh_rest;
  float* dL_dscales;
  float* dL_drotations;
  float* dL_dcov3D;
  float* dL_dface_center;
  float* dL_dface_orien_mat;
  float* dL_dface_scaling;
  /* Fused gradient all-reduce over NVLink/NVSwitch (BOUND_RAW mode, frame-sharded data parallel).  When 1, the six
   * parameter-gradient outputs (dL_dmeans3D, dL_drotations, dL_dscales, dL_dopacity, dL_dsh_dc, dL_dsh_rest) are
   * NVLS MULTICAST addresses of a symmetric buffer mapped on every rank of the group, and the kernel emits
   * multimem.red.add.f32 instead of stores: the switch sums the ranks' contributions while the backward kernel is
   * still running -- no separate all-reduce pass.  The caller zero-fills the buffer and barriers the group before
   * the call, and barriers again before reading the result (gaussianavatars_b200/dist.py does both).
   * Splats that received no gradient issue nothing (the buffer already holds their zero). */
  int32_t grads_are_multicast;
  /* Optional face-sorted view of `binding` (static between densifications, so the caller builds it once):
   * splats of one face are split into chunks (e.g. <= 16 splats); chunk c covers face_perm[face_chunk_start[c] ..
   * face_chunk_end[c]) and belongs to face face_chunk_face[c].  When given (num_face_chunks > 0), the face-frame
   * gradients are reduced per chunk by a second kernel instead of 13 global atomics per splat -- a face that owns
   * thousands of splats (hair, teeth) no longer serialises the L2 atomic unit. */
  const int32_t* face_perm;        /* [P] splat ids sorted by face */
  const int32_t* face_chunk_face;  /* [num_face_chunks] */
  const int32_t* face_chunk_start; /* [num_face_chunks] */
  const int32_t* face_chunk_end;   /* [num_face_chunks] */
  int32_t num_face_chunks;
} gab200_backward_args;

int32_t gab200_backward(const gab200_backward_args* args, void* stream);

/* Frustum test only.  Replaces diff_gaussian_rasterization._C.mark_visible (GaussianRasterizer.markVisible). */
int32_t gab200_mark_visible(int32_t P, const float* means3D, const float* viewmatrix, const float* projmatrix,
                            uint8_t* present /* [P] 0/1 */, void* stream);

/* Runs ONLY the binding + activation part of the fused preprocess (scene/gaussian_model.py:113-160) and exports
 * world-space means3D [P,3], opacities [P], scales [P,3] (exp * face scale) and cov3D [P,6] (with scale_modifier).
 * Any output may be NULL.  Same device code as the fused forward -> bit-identical values (parity tests, and the
 * callers that still need pc.get_xyz, e.g. convert_SHs_python). */
int32_t gab200_bind_activate(const gab200_forward_args* args, float* means3D, float* opacities, float* scales,
                             float* cov3D, void* stream);

/* Per-face frame of the posed mesh in one launch.  Replaces FlameGaussianModel.update_mesh_properties +
 * compute_face_orientation (scene/flame_gaussian_model.py:137-147, utils/graphics_utils.py:116-135):
 * verts [V,3], faces [F,3] int32 -> face_center [F,3], face_orien_mat [F,3,3] (columns a0 a1 a2), face_scaling [F]. */
int32_t gab200_face_frame_forward(int32_t F, int32_t V, const float* verts, const int32_t* faces, float* face_center,
                                  float* face_orien_mat, float* face_scaling, void* stream);
/* Its backward: dL/dverts [V,3] (zeroed by the library, then accumulated).  Any upstream gradient may be NULL (= 0). */
int32_t gab200_face_frame_backward(int32_t F, int32_t V, const float* verts, const int32_t* faces,
                                   const float* dL_dface_center, const float* dL_dface_orien_mat,
                                   const float* dL_dface_scaling, float* dL_dverts, void* stream);

/* FLAME head: blendshapes + linear blend skinning of one mesh per call, with its backward.  Replaces
 * FlameHead.forward(shape, expr, rotation, neck, jaw, eyes, translation, zero_centered_at_root_node=False,
 * return_landmarks=False, return_verts_cano=True, static_offset=...) and its autograd (flame_model/flame.py:485-558,
 * flame_model/lbs.py:25-57,101-304).  The model arrays are inputs (FlameHead's buffers in its layout; NB =
 * n_shape + n_expr); the caller precomputes J_template = J_regressor v_template and J_shapedirs = J_regressor shapedirs
 * once per model.  Per-timestep parameters are (T, k) tables read at the device row index `row` (NULL = row 0), so a
 * captured CUDA graph can replay any timestep; a row outside [0, T) turns every output of the call into NaN and the
 * backward into a no-op.  Forward: 2 launches, backward: 2 launches, no host synchronisation. */
typedef struct gab200_flame_args {
  uint32_t abi_version;
  int32_t V, n_shape, n_expr;
  int32_t J;                    /* joints: must be 5 (global, neck, jaw, left eye, right eye) */
  int32_t T;                    /* rows of the per-timestep tables */
  /* model */
  const float* v_template;      /* [V,3] */
  const float* shapedirs;       /* [V,3,NB] */
  const float* posedirs;        /* [(J-1)*9, V*3] */
  const float* J_regressor;     /* [J,V] dense */
  const float* lbs_weights;     /* [V,J] */
  const int32_t* parents;       /* [J] device; parents[j] in [0, j) for j >= 1 (otherwise the outputs are NaN) */
  const float* J_template;      /* [J,3] */
  const float* J_shapedirs;     /* [J,3,NB] */
  /* parameters */
  const int32_t* row;           /* device, one int32, or NULL (= row 0) */
  const float* shape;           /* [n_shape] or NULL (= 0) */
  const float* expr;            /* [T,n_expr] */
  const float* rotation;        /* [T,3] */
  const float* neck;            /* [T,3] */
  const float* jaw;             /* [T,3] */
  const float* eyes;            /* [T,6] */
  const float* translation;     /* [T,3] */
  const float* static_offset;   /* [V,3] or NULL (= 0) */
  /* outputs */
  float* verts;                 /* [V,3] */
  float* verts_cano;            /* [V,3] (v_shaped) or NULL */
  void* workspace;              /* gab200_flame_workspace_bytes(V, n_shape, n_expr) bytes, 256-byte aligned: written by the
                                   forward, read by the backward of the same call */
  /* gradients (backward): ADDED into; NULL = not wanted.  The (T,k) ones are touched in row `row` only.  Without
     grad_shape the shape columns of shapedirs (n_shape of NB) are not read. */
  float* grad_shape;            /* [n_shape] */
  float* grad_expr;             /* [T,n_expr] */
  float* grad_rotation;         /* [T,3] */
  float* grad_neck;             /* [T,3] */
  float* grad_jaw;              /* [T,3] */
  float* grad_eyes;             /* [T,6] */
  float* grad_translation;      /* [T,3] */
  float* grad_static_offset;    /* [V,3] */
} gab200_flame_args;
size_t gab200_flame_workspace_bytes(int32_t V, int32_t n_shape, int32_t n_expr);
int32_t gab200_flame_forward(const gab200_flame_args* args, void* stream);
/* dL_dverts [V,3]: gradient of the loss w.r.t. `verts` of the forward that filled args->workspace. */
int32_t gab200_flame_backward(const gab200_flame_args* args, const float* dL_dverts, void* stream);

/* Mean absolute error between a rendered image (n = 3*H*W floats) and a uint8 ground truth (value/255), with its
 * gradient, in one pass: *loss = mean |img - gt/255|, grad[i] = sign(img[i] - gt[i]/255) / n.  `loss` is zeroed by the
 * library.  Replaces `l1_loss(image, gt_image)` + its autograd and the float32 upload of the ground truth
 * (utils/loss_utils.py:17-18, train.py:128-131).  grad may be NULL (loss only). */
int32_t gab200_l1_loss_u8(int64_t n, const float* img, const uint8_t* gt, float* grad, float* loss, void* stream);
/* The gradient alone, scaled by an upstream gradient read from device memory (NULL = 1): grad[i] = *upstream *
 * sign(img[i] - gt[i]/255) / n.  What autograd's backward of the loss calls (grad may be NULL in the forward above:
 * loss only), so that no separate multiply pass runs over the (3,H,W) gradient. */
int32_t gab200_l1_loss_u8_backward(int64_t n, const float* img, const uint8_t* gt, const float* upstream, float* grad,
                                   void* stream);

/* Photometric training loss of the reference with its gradient, in two launches (SURVEY.md 8f rank 2):
 *   total = (1 - lambda_dssim) * mean|img - gt| + lambda_dssim * (1 - mean SSIM(img, gt))
 * Replaces `l1_loss(image, gt) * (1 - lambda)` + `(1 - ssim(image, gt)) * lambda` and their autograd
 * (utils/loss_utils.py:17-18,36-63; train.py:131-132): 11x11 Gaussian window, sigma 1.5, zero padding, C1 = 0.01^2,
 * C2 = 0.03^2, mean over all channels and pixels.  image / grad: float32 [channels, height, width]; gt: the same
 * shape as uint8 (value/255; gt_is_u8 = 1) or float32 (gt_is_u8 = 0).  loss[3] receives {L1 mean, SSIM mean, total}
 * scratch: GAB_PHOTOMETRIC_SCRATCH_HEAD + 3 * channels * height * width floats owned by the caller, 16-byte aligned
 * (two double accumulators, then the three partial-derivative maps handed from the first launch to the second). */
#define GAB_PHOTOMETRIC_SCRATCH_HEAD 4
typedef struct gab200_photometric_args {
  uint32_t abi_version;
  int32_t channels, height, width;
  int32_t gt_is_u8;
  float lambda_dssim;
  const float* image;
  const void* gt;
  float* grad;    /* [channels, height, width]  d total / d image */
  float* loss;    /* [3] */
  float* scratch; /* [GAB_PHOTOMETRIC_SCRATCH_HEAD + 3 * channels * height * width] */
} gab200_photometric_args;
int32_t gab200_photometric_loss(const gab200_photometric_args* args, void* stream);

/* Adam over several parameter arrays in one launch (SURVEY.md 8f rank 3).  Replaces `gaussians.optimizer.step()` for
 * the splat parameter groups (scene/gaussian_model.py:213-232 builds `torch.optim.Adam(l, lr=0.0, eps=1e-15)` with one
 * group -- and one learning rate -- per array; train.py:207-209): amsgrad off, no weight decay, bias-corrected, `step`
 * counts from 1.  `segments` is a HOST array; every pointer inside is a device pointer to n floats. */
#define GAB_ADAM_MAX_SEGMENTS 8 /* per launch; longer lists are split */
typedef struct gab200_adam_segment {
  float* param;
  const float* grad;
  float* exp_avg;
  float* exp_avg_sq;
  int64_t n;
  double lr; /* hyper-parameters travel as double, like the Python floats torch forms its scalars from */
} gab200_adam_segment;
int32_t gab200_adam_step(int32_t num_segments, const gab200_adam_segment* segments, int64_t step, double beta1,
                         double beta2, double eps, void* stream);

/* The position / scale regularisers of the mesh-bound training step (train.py:134-146), loss and gradient in one
 * launch each.  vis = radii > 0 of the frame just rendered.  loss[3] receives {xyz term, scale term, visible count};
 * sums: 3 doubles of device scratch shared by the forward and its backward.  The backward writes grad_xyz /
 * grad_scaling [P,3] in full (zeros for invisible splats) and ADDS into grad_face_scaling [F] (metric_* only; the
 * caller zero-fills it); g_out[2] = upstream gradients of the two terms (device). */
typedef struct gab200_regularize_args {
  uint32_t abi_version;
  int32_t P;
  int32_t metric_xyz, metric_scale;
  float threshold_xyz, threshold_scale, lambda_xyz, lambda_scale;
  const float *xyz, *scaling;          /* raw _xyz, _scaling [P,3] */
  const int32_t* radii;                /* [P] */
  const int32_t* binding;              /* [P] or NULL */
  const float* face_scaling;           /* [F] */
  float* loss;                         /* [3] */
  double* sums;                        /* [3] */
  float *grad_xyz, *grad_scaling, *grad_face_scaling;   /* backward only */
} gab200_regularize_args;
int32_t gab200_regularize_forward(const gab200_regularize_args* args, void* stream);
int32_t gab200_regularize_backward(const gab200_regularize_args* args, const float* g_out, void* stream);

/* In-place all-reduce (sum) of n floats that every rank of a group holds in NVLink symmetric memory, through the
 * NVSwitch multicast address `mc_ptr` of that allocation (NVLS): rank r reduces the r-th slice with
 * multimem.ld_reduce and stores it to every replica with multimem.st.  16-byte aligned.  The CALLER orders it between
 * two group barriers on the stream (every replica written before / every slice stored after): dist.py uses the
 * symmetric-memory signal pads.  Replaces the ncclAllReduce of the flat splat-gradient buffer (SURVEY.md 8e). */
int32_t gab200_nvls_allreduce(float* mc_ptr, int64_t n, int32_t rank, int32_t world, void* stream);

/* densify_and_prune of the splat arrays with the Adam-state surgery fused (SURVEY.md 8f rank 3).  Replaces
 * GaussianModel.densify_and_prune (scene/gaussian_model.py:503-519 -> densify_and_clone :481-501, densify_and_split
 * :451-479, prune_points :371-397) together with the optimizer surgery it drives (:334-369, :399-424) and the
 * binding / binding_counter bookkeeping (:375-380, :395-397, :472-474, :495-497).  Two calls, because the caller has to
 * size the outputs:
 *   gab200_densify_plan   classifies every splat and scans the result; performs ONE stream synchronisation and leaves
 *                         totals_host = {kept originals, kept clones, kept child pairs, split parents}.
 *                         Output rows: P' = totals[0] + totals[1] + 2 * totals[2], in the reference's order
 *                         (originals, clones, first children, second children).
 *   gab200_densify_apply  gathers the six parameter arrays and their exp_avg / exp_avg_sq into the outputs (new rows get
 *                         zero moments), samples the children (noise: [2 * totals[3], 3] STANDARD normal values, rows
 *                         [0, S) for the first child of the S split parents in index order, [S, 2S) for the second --
 *                         exactly what torch.normal(mean=0, std=...) draws), and rebuilds binding / binding_counter.
 * The densification statistics (xyz_gradient_accum, denom, max_radii2D) of the result are all zero in the reference
 * (densification_postfix :447-449): the caller allocates zeros of length P'. */
typedef struct gab200_densify_args {
  uint32_t abi_version;
  int32_t P, num_faces;
  int32_t sh_rest_width;   /* floats per splat of _features_rest: 3 * (M - 1) */
  float grad_threshold, min_opacity, extent, percent_dense;
  float max_screen_size;   /* <= 0: None */
  const float *xyz, *rotation, *scaling, *opacity, *f_dc, *f_rest;   /* raw parameters [P, 3|4|3|1|3|sh_rest_width] */
  const float* exp_avg[6];     /* Adam moments in the order xyz, rotation, scaling, opacity, f_dc, f_rest; NULL = none */
  const float* exp_avg_sq[6];
  const float *xyz_gradient_accum, *denom;   /* [P] */
  const int32_t* binding;          /* [P] or NULL (plain GaussianModel) */
  const int32_t* binding_counter;  /* [F] */
  const float* face_scaling;       /* [F] */
  void* scratch;                   /* device, gab200_densify_scratch_bytes(P, F) bytes, 256-byte aligned; shared by both calls */
  uint32_t* totals_host;           /* HOST (pinned), 4 words */
} gab200_densify_args;
typedef struct gab200_densify_out {
  int32_t P_out, n_child_rows;     /* totals[0] + totals[1] + 2 totals[2];  2 totals[2] */
  float *xyz, *rotation, *scaling, *opacity, *f_dc, *f_rest;
  float* exp_avg[6];
  float* exp_avg_sq[6];
  int32_t* binding;                /* [P_out] or NULL */
  int32_t* binding_counter;        /* [F] or NULL */
  const float* noise;              /* [2 * totals[3], 3] */
  int32_t* src_scratch;            /* [P_out] device scratch */
  uint8_t* kind_scratch;           /* [P_out] */
  int32_t* noise_row_scratch;      /* [totals[2]] */
} gab200_densify_out;
size_t gab200_densify_scratch_bytes(int32_t P, int32_t num_faces);
int32_t gab200_densify_plan(const gab200_densify_args* args, void* stream);
int32_t gab200_densify_apply(const gab200_densify_args* args, const gab200_densify_out* out, void* stream);

/* Debug/parity access to a finished forward: copies the sorted (key,value) stream and tile ranges to caller
 * DEVICE buffers: keys [N] u64, values [N] u32, ranges [tiles,2] u32. Any may be NULL. */
int32_t gab200_export_binning(const gab200_forward_args* args, const gab200_frame_state* state, uint64_t* keys,
                              uint32_t* values, uint32_t* ranges, void* stream);

/* Opt-in per-stage device timing (profiling aid used by bench.py's roofline line).  When enabled, forward/backward
 * bracket every stage with cudaEvents on the launching stream.  gab200_stage_times() synchronises the pending
 * events, adds them to per-stage totals and returns totals (milliseconds) and launch counts since the last reset. */
enum {
  GAB200_STAGE_PREPROCESS = 0,
  GAB200_STAGE_SCAN = 1,
  GAB200_STAGE_EMIT_KEYS = 2,
  GAB200_STAGE_SORT = 3,
  GAB200_STAGE_TILE_RANGES = 4,
  GAB200_STAGE_BLEND_FWD = 5,
  GAB200_STAGE_BLEND_BWD = 6,
  GAB200_STAGE_PREPROCESS_BWD = 7,
  GAB200_NUM_STAGES = 8
};
void gab200_stage_timing_enable(int32_t enable);
/* Host-side wall time (microseconds, accumulated since the last reset) spent inside gab200_forward, split into
 * [0] launches before the sync, [1] waiting for N, [2] binning allocation callback(s), [3] emit+sort+ranges dispatch,
 * [4] blend dispatch, [5] number of forwards.  Profiling aid; always on (a few clock reads per call). */
void gab200_host_times(double out[6], int32_t reset);
int32_t gab200_stage_times(double total_ms[GAB200_NUM_STAGES], int64_t launches[GAB200_NUM_STAGES], int32_t reset);

/* Tuning knobs (process-wide, atomics; every value has a built-in default that suits the headline workload).
 * gab200_tune(knob, value) sets a knob and returns the previous value; value < 0 only queries. */
enum {
  GAB200_TUNE_HEAVY_FWD = 0,   /* forward blend: a tile is "heavy" (1 px/thread, 8 warps) from this list length (default 32) */
  GAB200_TUNE_HEAVY_BWD = 1,   /* backward blend: a tile is "heavy" (K = 2, 4 warps) from this list length (default 2048) */
  GAB200_TUNE_DEPTH_SORT = 2,  /* 0 (default): bucket sort when a depth hint is given; 1: always cub radix sort */
  GAB200_TUNE_BWD_VARIANT = 3, /* backward blend schedule (same arithmetic, same results up to summation order):
                                  0 tile = CTA group, live-band-set specialised bodies; 1 warp-independent tasks,
                                  straight-line bands, pipelined reduction; 2 / 3 as 1 with dead bands skipped by
                                  uniform branches always / unless all bands are live; 4, 5 = 3, 2 compiled for 5 CTAs
                                  per SM; 6 = 1 with specialised bodies; 7 = 2 for 6 CTAs per SM; 8 (default) = 3 with
                                  the two bands of a pair in packed fp32x2 arithmetic (FFMA2 / FMUL2 / FADD2); 9 = 8
                                  for 5 CTAs per SM.  Measured at the headline size (profiles/r02/bwd_variants.jsonl,
                                  bwd_packed_variants.jsonl): 211 / 198 / 179 / 175 / 182 / 185 / 186 / 211 / 171 /
                                  196 us */
  GAB200_TUNE_TILE_SORT = 4,   /* per-instance sort by tile: 0 (default) cub::DeviceRadixSort::SortPairs over the instances
                                  (5 launches + tile-range detection); 1 counting sort by tile + per-tile rank sort
                                  (csrc/tile_sort.cu: 3 launches, no memsets).  Identical sorted streams; at the headline
                                  size the counting form is SLOWER (same-address atomics on the hot tiles' counters:
                                  preprocess +18 us, emission 26 -> 78 us; profiles/r02/tile_sort_counting_vs_cub.json) */
  GAB200_TUNE_NVLS_CTAS = 5,   /* gab200_nvls_allreduce: CTAs of 256 threads (0 = default: 64) */
  GAB200_NUM_TUNABLES = 8
};
int32_t gab200_tune(int32_t knob, int32_t value);

/* Number of kernels launched by this library on the calling process so far (bench.py's gpu_launches claim). */
int64_t gab200_launch_count(void);

const char* gab200_status_string(int32_t status);
uint32_t gab200_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* GAB200_RASTERIZER_H */
