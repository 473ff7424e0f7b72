// api.cu -- the extern "C" boundary declared in include/gab200_rasterizer.h.  Host orchestration only: argument
// validation, carving of the three caller-allocated byte buffers, stage launches, and the policy for learning the
// instance count N (gab200_sync_mode: a wait in the middle, a wait at the end that normally finds its answer ready,
// or no wait at all under CUDA-graph capture).  No torch types, no exceptions; process-wide state is limited to
// atomics (launch counter, profiling timers, tuning knobs).
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

#include "common.cuh"
#include "kernels.cuh"

namespace gab {
static std::atomic<int64_t> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

// cub's temp-storage queries run its whole host-side dispatch; the answer only grows with N -> cache it.
struct SortTempCache {
  int64_t n = -1;
  int bits = -1;
  size_t bytes = 0;
};
static thread_local SortTempCache t_sort_cache[2];  // [0]: stage A (32-bit depth keys), [1]: stage B (tile ids)
static size_t cached_sort_temp_bytes(int64_t N, int bits) {
  SortTempCache& c = t_sort_cache[bits == 32 ? 0 : 1];
  if (c.bits != bits || N > c.n) {
    const int64_t n_up = N + N / 2 + 1024;  // headroom so that the query is rare
    c.bytes = sort_temp_bytes(n_up, bits);
    c.n = n_up;
    c.bits = bits;
  }
  return c.bytes;
}

struct GeomView {
  SplatRec* rec;
  SplatAux* aux;
  uint32_t* tiles_touched;
  uint32_t* offsets;
  uint8_t* clamped;
  uint32_t* depth_keys[2];  // stage-A sort: fp32 depth bit patterns (double buffer)
  uint32_t* ids[2];         //               splat ids (double buffer) -> depth order
  void* sortA_temp;
  size_t sortA_temp_bytes;
  float* g2d;
  float* face_scratch;  // [P,13] per-splat face-frame gradients (CSR route of the fused backward)
  void* scan_temp;
  size_t scan_temp_bytes;
  DepthBuckets buckets;  // bucket-sort bookkeeping (counts | tiles | meta contiguous: one memset)
  size_t bucket_clear_bytes;
  size_t bytes;
};
// buckets for the per-splat depth sort: 32..64 splats each, a power of two in [256, 8192]
static uint32_t depth_bucket_count(int P) {
  uint32_t nb = 256;
  while (nb < 8192 && (int64_t)nb * 64 < P) nb <<= 1;
  return nb;
}
// The layout is a pure function of (P, need_backward): the only size that depends on anything else (cub's temp
// storage for the stage-A radix sort, `sort_temp`) is carved LAST, so the backward -- which passes 0 for it, on
// whatever host thread autograd picked -- sees every other array at the forward's offset.
static GeomView carve_geom(void* base, int P, bool need_backward, size_t sort_temp) {
  GeomView g;
  Carver c(base);
  g.rec = c.take<SplatRec>((size_t)P);
  g.aux = c.take<SplatAux>((size_t)P);
  g.tiles_touched = c.take<uint32_t>((size_t)P);
  g.offsets = c.take<uint32_t>((size_t)P);
  g.clamped = c.take<uint8_t>((size_t)P);
  g.depth_keys[0] = c.take<uint32_t>((size_t)P);
  g.depth_keys[1] = c.take<uint32_t>((size_t)P);
  g.ids[0] = c.take<uint32_t>((size_t)P);
  g.ids[1] = c.take<uint32_t>((size_t)P);
  g.g2d = need_backward ? c.take<float>((size_t)P * GAB_G2D_STRIDE) : nullptr;
  g.face_scratch = need_backward ? c.take<float>((size_t)P * GAB_FACE_GRAD_STRIDE) : nullptr;
  g.scan_temp_bytes = scan_temp_bytes(P);
  g.scan_temp = c.take<char>(g.scan_temp_bytes);
  {
    DepthBuckets& d = g.buckets;
    d.nb = depth_bucket_count(P);
    uint32_t* head = c.take<uint32_t>((size_t)2 * d.nb + GAB_DEPTH_META_WORDS);
    d.counts = head;
    d.tiles = head ? head + d.nb : nullptr;
    d.meta = head ? head + 2 * d.nb : nullptr;
    g.bucket_clear_bytes = sizeof(uint32_t) * ((size_t)2 * d.nb + GAB_DEPTH_META_WORDS);
    d.start = c.take<uint32_t>((size_t)d.nb);
    d.tile_base = c.take<uint32_t>((size_t)d.nb);
    d.rank = c.take<uint32_t>((size_t)P);
    d.lo = d.hi = 0;
    d.scale = 0.f;
    d.enabled = 0;
  }
  g.sortA_temp_bytes = sort_temp;
  g.sortA_temp = c.take<char>(sort_temp);
  g.bytes = c.bytes();
  return g;
}
struct BinView {
  uint32_t* keys[2];  // tile ids (stage-B sort keys)
  uint32_t* vals[2];  // splat ids
  uint8_t* strip_mask;  // per sorted instance: which 16x2 pixel strips of its tile it contributed to (forward -> backward)
  void* sort_temp;
  size_t sort_temp_bytes;
  size_t bytes;
};
static BinView carve_binning(void* base, int64_t N, bool need_backward, size_t sort_temp) {
  BinView b;
  Carver c(base);
  // + 320: the blend kernels fetch id lists with 16-B-granular bulk copies of up to 256+4 ids that may start
  // 3 ids before a tile's run and end past the stream's last id; the slack keeps those reads inside the buffer
  const size_t n = (size_t)(N > 0 ? N : 1) + 320;
  b.keys[0] = c.take<uint32_t>(n);
  b.keys[1] = c.take<uint32_t>(n);
  b.vals[0] = c.take<uint32_t>(n);
  b.vals[1] = c.take<uint32_t>(n);
  b.strip_mask = need_backward ? c.take<uint8_t>(n) : nullptr;
  b.sort_temp_bytes = sort_temp;
  b.sort_temp = c.take<char>(sort_temp);
  b.bytes = c.bytes();
  return b;
}
struct ImageView {
  uint2* ranges;
  uint32_t* order;
  uint32_t* order_info;
  uint32_t* tile_count;   // counting tile sort: instances per tile (RED by preprocess), zeroed before it
  uint32_t* tile_cursor;  //                     next free slot of the tile's segment (emission)
  float* final_T;
  uint32_t* n_contrib;
  size_t bytes;
};
static ImageView carve_image(void* base, int W, int H, bool need_backward) {
  ImageView v;
  Carver c(base);
  const int gx = (W + GAB_TILE - 1) / GAB_TILE, gy = (H + GAB_TILE - 1) / GAB_TILE;
  v.ranges = c.take<uint2>((size_t)gx * gy + 1);  // + 1: the slot the sentinel key of a capacity-padded sort maps to
  v.order = c.take<uint32_t>((size_t)gx * gy);
  v.order_info = c.take<uint32_t>(4);
  v.tile_count = c.take<uint32_t>((size_t)gx * gy);
  v.tile_cursor = c.take<uint32_t>((size_t)gx * gy);
  v.final_T = need_backward ? c.take<float>((size_t)W * H) : nullptr;
  v.n_contrib = need_backward ? c.take<uint32_t>((size_t)W * H) : nullptr;
  v.bytes = c.bytes();
  return v;
}

// ---- opt-in stage timing -------------------------------------------------------------------------------
struct StageTimer {
  std::atomic<int> enabled{0};
  std::mutex mu;
  struct Pending { int stage; cudaEvent_t a, b; };
  std::vector<Pending> pending;
  std::vector<cudaEvent_t> pool;
  double total_ms[GAB200_NUM_STAGES] = {0};
  int64_t launches[GAB200_NUM_STAGES] = {0};
  cudaEvent_t get() {
    if (!pool.empty()) { cudaEvent_t e = pool.back(); pool.pop_back(); return e; }
    cudaEvent_t e; cudaEventCreate(&e); return e;
  }
};
static StageTimer g_timer;
static thread_local bool t_capturing = false;  // the calling thread's stream is being captured: no timing events
struct StageScope {
  int stage; cudaStream_t stream; cudaEvent_t a{}, b{}; bool on;
  StageScope(int st, cudaStream_t s) : stage(st), stream(s), on(g_timer.enabled.load() != 0 && !t_capturing) {
    if (on) {
      std::lock_guard<std::mutex> l(g_timer.mu);
      a = g_timer.get(); b = g_timer.get();
      cudaEventRecord(a, stream);
    }
  }
  ~StageScope() {
    if (on) {
      cudaEventRecord(b, stream);
      std::lock_guard<std::mutex> l(g_timer.mu);
      g_timer.pending.push_back({stage, a, b});
    }
  }
};

// host-side profile of gab200_forward (nanoseconds, relaxed atomics: any thread may run a forward)
static std::atomic<int64_t> g_host_ns[6];
static inline void host_add(int i, double us) { g_host_ns[i].fetch_add((int64_t)(us * 1e3), std::memory_order_relaxed); }
static inline double now_us() {
  return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// N is read back through a pinned slot + event spin: lower wake-up latency than cudaStreamSynchronize and it only
// waits for the copy, not for anything the caller may have queued behind it on other streams.
struct PinnedSlot {
  uint32_t* host = nullptr;
  cudaEvent_t ev = nullptr;
  bool ok() {
    if (host == nullptr) {
      if (cudaHostAlloc((void**)&host, 64, cudaHostAllocDefault) != cudaSuccess) return false;
      if (cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess) return false;
    }
    return true;
  }
};
static thread_local PinnedSlot t_slot;

static int check_arch() {
  constexpr int MAX_DEV = 64;
  static std::atomic<int> cached[MAX_DEV];  // per device: 0 unknown, 1 ok, -1 bad
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return -1;
  const bool slot = dev >= 0 && dev < MAX_DEV;
  int c = slot ? cached[dev].load(std::memory_order_relaxed) : 0;
  if (c != 0) return c;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return -1;
  c = (major == 10) ? 1 : -1;
  if (slot) cached[dev].store(c, std::memory_order_relaxed);
  return c;
}

// tuning knobs (gab200_tune)
static std::atomic<int> g_tune[GAB200_NUM_TUNABLES];
static const int g_tune_default[GAB200_NUM_TUNABLES] = {32, 2048, 0, 8, 0, 0, 0, 0};  // see GAB200_TUNE_*
int tune_get(int knob) {
  const int v = g_tune[knob].load(std::memory_order_relaxed);
  return v > 0 ? v - 1 : g_tune_default[knob];  // stored biased by one so that zero-initialised = "default"
}

static bool validate(const gab200_forward_args* a) {
  if (a == nullptr || a->abi_version != GAB200_ABI_VERSION) return false;
  if (a->P < 0 || a->image_width <= 0 || a->image_height <= 0) return false;
  if (a->out_color == nullptr || (a->P > 0 && a->radii == nullptr)) return false;
  if (!a->bg || !a->viewmatrix || !a->projmatrix || !a->campos) return false;
  if (!a->alloc_geom || !a->alloc_binning || !a->alloc_image) return false;
  if (a->P == 0) return true;
  if (!a->means3D || !a->opacities) return false;
  if (a->sh_degree < 0 || a->sh_degree > 3) return false;
  const int nb = (a->sh_degree + 1) * (a->sh_degree + 1);
  if (a->input_mode == GAB200_INPUT_ACTIVATED) {
    const bool has_sr = a->scales != nullptr && a->rotations != nullptr;
    if (has_sr == (a->cov3D_precomp != nullptr)) return false;  // exactly one of (scale,rot) / cov3D
    if ((a->scales != nullptr) != (a->rotations != nullptr)) return false;
    if ((a->shs != nullptr) == (a->colors_precomp != nullptr)) return false;  // exactly one of SH / colours
    if (a->shs != nullptr && a->sh_coeffs < nb) return false;
  } else if (a->input_mode == GAB200_INPUT_BOUND_RAW) {
    if (!a->scales || !a->rotations || a->cov3D_precomp) return false;
    if (a->colors_precomp == nullptr) {
      if (!a->sh_dc || a->sh_coeffs < nb) return false;
      if (a->sh_coeffs > 1 && !a->sh_rest) return false;
    }
    if (a->binding != nullptr && (!a->face_center || !a->face_orien_mat || !a->face_scaling || a->num_faces <= 0))
      return false;
  } else {
    return false;
  }
  return true;
}

#define GAB_CUDA(expr)                                  \
  do {                                                  \
    cudaError_t _e = (expr);                            \
    if (_e != cudaSuccess) return GAB200_ERR_CUDA;      \
  } while (0)
#define GAB_STAGE_CHECK(dbg, stream)                                  \
  do {                                                                \
    if (cudaPeekAtLastError() != cudaSuccess) return GAB200_ERR_CUDA; \
    if (dbg) GAB_CUDA(cudaStreamSynchronize(stream));                 \
  } while (0)

}  // namespace gab

using namespace gab;

extern "C" {

uint32_t gab200_abi_version(void) { return GAB200_ABI_VERSION; }

void gab200_stage_timing_enable(int32_t enable) { g_timer.enabled.store(enable ? 1 : 0); }

int32_t gab200_stage_times(double total_ms[GAB200_NUM_STAGES], int64_t launches[GAB200_NUM_STAGES], int32_t reset) {
  std::lock_guard<std::mutex> l(g_timer.mu);
  for (auto& p : g_timer.pending) {
    if (cudaEventSynchronize(p.b) != cudaSuccess) return GAB200_ERR_CUDA;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, p.a, p.b) != cudaSuccess) return GAB200_ERR_CUDA;
    g_timer.total_ms[p.stage] += ms;
    g_timer.launches[p.stage] += 1;
    g_timer.pool.push_back(p.a);
    g_timer.pool.push_back(p.b);
  }
  g_timer.pending.clear();
  for (int i = 0; i < GAB200_NUM_STAGES; i++) {
    if (total_ms) total_ms[i] = g_timer.total_ms[i];
    if (launches) launches[i] = g_timer.launches[i];
    if (reset) { g_timer.total_ms[i] = 0; g_timer.launches[i] = 0; }
  }
  return GAB200_OK;
}
int64_t gab200_launch_count(void) { return g_launches.load(); }

void gab200_host_times(double out[6], int32_t reset) {
  for (int i = 0; i < 6; i++) {
    const int64_t v = reset ? g_host_ns[i].exchange(0) : g_host_ns[i].load();
    if (out) out[i] = i == 5 ? (double)v : (double)v * 1e-3;
  }
}

int32_t gab200_tune(int32_t knob, int32_t value) {
  if (knob < 0 || knob >= GAB200_NUM_TUNABLES) return GAB200_ERR_INVALID_ARGUMENT;
  const int prev = tune_get(knob);
  if (value >= 0) g_tune[knob].store(value + 1, std::memory_order_relaxed);
  return prev;
}

int32_t gab200_counters_ok(const uint32_t* c, uint32_t frame_seq) {
  if (c == nullptr) return GAB200_ERR_INVALID_ARGUMENT;
  const volatile uint32_t* v = c;
  if (v[GAB200_CTR_SEQ] != frame_seq) return -1;
  return (v[GAB200_CTR_NUM_RENDERED_HI] == 0 && v[GAB200_CTR_BUCKET_OVERFLOW] == 0 &&
          v[GAB200_CTR_NUM_RENDERED] <= v[GAB200_CTR_CAPACITY]) ? 1 : 0;
}

const char* gab200_status_string(int32_t s) {
  switch (s) {
    case GAB200_OK: return "ok";
    case GAB200_ERR_INVALID_ARGUMENT: return "invalid argument (shape / missing pointer / inconsistent options)";
    case GAB200_ERR_CUDA: return "CUDA runtime or kernel error";
    case GAB200_ERR_ALLOC: return "allocation callback returned NULL";
    case GAB200_ERR_ARCH: return "device is not sm_100 class (this library ships sm_100a code only)";
    case GAB200_ERR_OVERFLOW: return "instance count overflows 32 bits";
    default: return "unknown status";
  }
}

// ---- forward, in pieces ----------------------------------------------------------------------------------
namespace {
struct Frame {
  const gab200_forward_args* a;
  gab200_frame_state* st;
  cudaStream_t stream;
  GeomView g;
  ImageView iv;
  int P, W, H, gx, gy;
  bool nb, dbg;
  uint32_t* ctr_host;   // where the counters land on the host
  cudaEvent_t ctr_event;
  int selA = 0;                           // which half of the stage-A double buffer holds the depth order
  const uint32_t* order_count = nullptr;  // device count of listed splats (bucket path), else all P are listed
  bool counting = true;                   // tile sort: counting sort + per-tile rank sort (tile_sort.cu), else cub radix
  uint32_t scan_clamp = 0xffffffffu;      // capacity the tile ranges were cut at by the last tile scan
};

// preprocess (+ bucket bookkeeping when `bucket`) -> per-splat depth order + emission offsets -> counters published
// on the device and copied to the host slot, event recorded behind the copy.
int enqueue_geometry(Frame& f, bool bucket, bool run_preprocess, uint32_t capacity) {
  const gab200_forward_args* a = f.a;
  GeomView& g = f.g;
  cudaStream_t stream = f.stream;
  DepthBuckets& d = g.buckets;
  d.enabled = 0;
  if (bucket) {
    d.lo = a->depth_hint_lo;
    d.hi = a->depth_hint_hi;
    d.scale = (float)((double)d.nb / ((double)(d.hi - d.lo) + 1.0));
    d.enabled = 1;
  }
  const int tiles = f.gx * f.gy;
  if (run_preprocess) {
    GAB_CUDA(cudaMemsetAsync(d.counts, 0, g.bucket_clear_bytes, stream));
    if (f.counting) GAB_CUDA(cudaMemsetAsync(f.iv.tile_count, 0, sizeof(uint32_t) * (size_t)tiles, stream));
    StageScope sc(GAB200_STAGE_PREPROCESS, stream);
    launch_preprocess(*a, g.rec, g.aux, g.tiles_touched, f.nb ? g.clamped : nullptr, g.depth_keys[0], g.ids[0], g.buckets,
                      f.counting ? f.iv.tile_count : nullptr, stream);
  }
  GAB_STAGE_CHECK(f.dbg, stream);
  if (f.counting && run_preprocess) {
    // tile ranges, write cursors, N and the heaviest-first tile order straight from the per-tile counts
    StageScope sc(GAB200_STAGE_TILE_RANGES, stream);
    f.scan_clamp = capacity > 0 ? capacity : 0xffffffffu;
    launch_tile_scan_order(tiles, f.iv.tile_count, f.scan_clamp, f.iv.ranges, f.iv.tile_cursor, f.iv.order,
                           f.iv.order_info, g.buckets.meta, tune_get(GAB200_TUNE_HEAVY_FWD),
                           tune_get(GAB200_TUNE_HEAVY_BWD), stream);
  }
  {
    StageScope sc(GAB200_STAGE_SCAN, stream);
    if (bucket) {
      // per-splat depth order + emission offsets as a bucket sort over the hinted key range -- see binning.cu
      launch_depth_bucket_sort(f.P, g.buckets, g.depth_keys[0], g.tiles_touched, g.depth_keys[1], g.ids[1], g.offsets,
                               capacity, a->frame_seq, a->sync_mode == GAB200_SYNC_NONE ? a->overflow_flag : nullptr,
                               stream);
      f.selA = 1;
      f.order_count = g.buckets.meta + GAB200_CTR_NUM_LISTED;
    } else {
      // stage A of the key sort (per splat, by depth) + emission offsets in depth order  -- see binning.cu
      GAB_CUDA(run_sort(g.sortA_temp, g.sortA_temp_bytes, g.depth_keys[0], g.depth_keys[1], g.ids[0], g.ids[1], f.P, 32,
                        &f.selA, stream));
      if (!f.counting)  // emission offsets in depth order: only the radix tile sort places instances by them
        GAB_CUDA(run_scan(g.scan_temp, g.scan_temp_bytes, g.ids[f.selA], g.tiles_touched, g.offsets, f.P, stream));
      f.order_count = nullptr;
    }
    if (!bucket)
      launch_publish_counters(g.buckets.meta, f.counting ? nullptr : g.offsets, f.P, capacity, a->frame_seq,
                              a->sync_mode == GAB200_SYNC_NONE ? a->overflow_flag : nullptr, stream);
  }
  GAB_STAGE_CHECK(f.dbg, stream);
  GAB_CUDA(cudaMemcpyAsync(f.ctr_host, g.buckets.meta, sizeof(uint32_t) * GAB200_NUM_COUNTERS, cudaMemcpyDeviceToHost,
                           stream));
  if (f.ctr_event) GAB_CUDA(cudaEventRecord(f.ctr_event, stream));
  return GAB200_OK;
}

// emit -> per-instance tile sort -> ranges -> tile order -> blend, for a binning buffer of `cap` instances.
// n_known >= 0: exactly that many instances exist (no padding); n_known < 0: the count is only on the device -- the
// tile sort runs over the whole capacity, unused slots carry the sentinel key and sort behind every tile.
int enqueue_binning_blend(Frame& f, void* bin, int64_t cap, int64_t n_known, size_t sort_temp, bool redo) {
  const gab200_forward_args* a = f.a;
  gab200_frame_state* st = f.st;
  cudaStream_t stream = f.stream;
  const int tiles = f.gx * f.gy;
  BinView bv = carve_binning(bin, cap, f.nb, sort_temp);
  st->binning_capacity = cap;
  st->binning_buffer = bin;
  st->binning_bytes = bv.bytes;
  const int64_t n_sort = n_known >= 0 ? n_known : cap;
  const bool counting = f.counting && f.P > 0;
  st->tile_sort_path = counting ? 1 : 0;
  if (bv.strip_mask != nullptr && n_sort > 0) GAB_CUDA(cudaMemsetAsync(bv.strip_mask, 0, (size_t)n_sort, stream));
  int selector = 0;
  if (counting) {
    if (redo) {  // the cursors were consumed (and the ranges possibly cut at a smaller capacity) by the first attempt
      StageScope sc(GAB200_STAGE_TILE_RANGES, stream);
      f.scan_clamp = (uint32_t)(cap < 0xffffffffll ? cap : 0xffffffffll);
      launch_tile_scan_order(tiles, f.iv.tile_count, f.scan_clamp, f.iv.ranges, f.iv.tile_cursor, f.iv.order,
                             f.iv.order_info, f.g.buckets.meta, tune_get(GAB200_TUNE_HEAVY_FWD),
                             tune_get(GAB200_TUNE_HEAVY_BWD), stream);
    }
    if (n_sort > 0) {
      {
        StageScope sc(GAB200_STAGE_EMIT_KEYS, stream);
        launch_emit_keys(f.P, f.gx, f.gy, f.g.rec, f.g.aux, f.g.ids[f.selA], nullptr, f.order_count, f.g.buckets.meta,
                         (uint32_t)cap, f.iv.tile_cursor, bv.keys[0], bv.vals[0], a->exact_binning, stream);
      }
      GAB_STAGE_CHECK(f.dbg, stream);
      {
        StageScope sc(GAB200_STAGE_SORT, stream);
        launch_tile_sort(tiles, f.iv.ranges, f.iv.order, f.iv.order_info, bv.keys[0], bv.vals[0], f.g.ids[f.selA],
                         f.order_count, f.P, stream);
      }
      GAB_STAGE_CHECK(f.dbg, stream);
    }
  } else {
    GAB_CUDA(cudaMemsetAsync(f.iv.ranges, 0, sizeof(uint2) * ((size_t)tiles + 1), stream));
    if (n_sort > 0) {
      if (n_known < 0) GAB_CUDA(cudaMemsetAsync(bv.keys[0], 0xff, sizeof(uint32_t) * (size_t)cap, stream));
      {
        StageScope sc(GAB200_STAGE_EMIT_KEYS, stream);
        launch_emit_keys(f.P, f.gx, f.gy, f.g.rec, f.g.aux, f.g.ids[f.selA], f.g.offsets, f.order_count, f.g.buckets.meta,
                         (uint32_t)cap, nullptr, bv.keys[0], bv.vals[0], a->exact_binning, stream);
      }
      GAB_STAGE_CHECK(f.dbg, stream);
      {
        StageScope sc(GAB200_STAGE_SORT, stream);
        GAB_CUDA(run_sort(bv.sort_temp, bv.sort_temp_bytes, bv.keys[0], bv.keys[1], bv.vals[0], bv.vals[1], n_sort,
                          st->sort_bits, &selector, stream));
      }
      GAB_STAGE_CHECK(f.dbg, stream);
      {
        StageScope sc(GAB200_STAGE_TILE_RANGES, stream);
        launch_tile_ranges(n_sort, (uint32_t)tiles, bv.keys[selector], f.iv.ranges, stream);
      }
      GAB_STAGE_CHECK(f.dbg, stream);
    }
    StageScope sc(GAB200_STAGE_TILE_RANGES, stream);
    launch_tile_scan_order(tiles, nullptr, 0xffffffffu, f.iv.ranges, nullptr, f.iv.order, f.iv.order_info, nullptr,
                           tune_get(GAB200_TUNE_HEAVY_FWD), tune_get(GAB200_TUNE_HEAVY_BWD), stream);
  }
  st->sorted_selector = selector;
  {
    StageScope sc(GAB200_STAGE_BLEND_FWD, stream);
    launch_blend_forward(f.W, f.H, f.iv.ranges, f.iv.order, f.iv.order_info, bv.vals[selector], f.g.rec, a->bg,
                         a->out_color, f.iv.final_T, f.iv.n_contrib, bv.strip_mask, stream);
  }
  GAB_STAGE_CHECK(f.dbg, stream);
  return GAB200_OK;
}

int wait_counters(Frame& f) {
  for (;;) {
    const cudaError_t q = cudaEventQuery(f.ctr_event);
    if (q == cudaSuccess) return GAB200_OK;
    if (q != cudaErrorNotReady) return GAB200_ERR_CUDA;
  }
}
}  // namespace

int64_t gab200_forward(const gab200_forward_args* a, gab200_frame_state* st, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (!validate(a) || st == nullptr) return GAB200_ERR_INVALID_ARGUMENT;
  if (check_arch() < 0) return GAB200_ERR_ARCH;
  memset(st, 0, sizeof(*st));
  Frame f;
  f.a = a; f.st = st; f.stream = stream;
  f.P = a->P; f.W = a->image_width; f.H = a->image_height;
  f.gx = (f.W + GAB_TILE - 1) / GAB_TILE; f.gy = (f.H + GAB_TILE - 1) / GAB_TILE;
  f.nb = a->need_backward != 0;
  f.dbg = a->debug != 0;
  f.counting = tune_get(GAB200_TUNE_TILE_SORT) == 1;
  const int P = f.P;
  const int mode = a->sync_mode;
  const bool speculative = mode != GAB200_SYNC_EXACT;  // binning + blend are enqueued before N is known
  if (speculative && P > 0 && a->binning_hint <= 0) return GAB200_ERR_INVALID_ARGUMENT;
  if (mode == GAB200_SYNC_NONE && a->counters_host == nullptr) return GAB200_ERR_INVALID_ARGUMENT;
  cudaStreamCaptureStatus cap_status = cudaStreamCaptureStatusNone;
  GAB_CUDA(cudaStreamIsCapturing(stream, &cap_status));
  if (cap_status != cudaStreamCaptureStatusNone && mode != GAB200_SYNC_NONE) return GAB200_ERR_INVALID_ARGUMENT;
  struct CaptureGuard {
    bool prev;
    explicit CaptureGuard(bool c) : prev(t_capturing) { t_capturing = c; }
    ~CaptureGuard() { t_capturing = prev; }
  } capture_guard(cap_status != cudaStreamCaptureStatusNone);

  // ---- geometry + image buffers ----
  const size_t tempA = cached_sort_temp_bytes(P > 0 ? P : 1, 32);
  GeomView gsz = carve_geom(nullptr, P, f.nb, tempA);
  void* geom = a->alloc_geom(a->alloc_user, gsz.bytes);
  if (geom == nullptr) return GAB200_ERR_ALLOC;
  f.g = carve_geom(geom, P, f.nb, tempA);
  ImageView isz = carve_image(nullptr, f.W, f.H, f.nb);
  void* img = a->alloc_image(a->alloc_user, isz.bytes);
  if (img == nullptr) return GAB200_ERR_ALLOC;
  f.iv = carve_image(img, f.W, f.H, f.nb);
  st->geom_buffer = geom; st->geom_bytes = f.g.bytes;
  st->image_buffer = img; st->image_bytes = f.iv.bytes;
  st->sort_bits = (int)tile_bits((uint32_t)(f.gx * f.gy));  // stage B: tile id only
  st->depth_bits = 32;                                      // stage A: the full fp32 depth pattern
  st->device_counters = f.g.buckets.meta;
  st->attempts = 1;
  st->depth_key_min = 1; st->depth_key_max = 0;  // "nothing visible" until the counters say otherwise

  const double t0 = now_us();
  if (P == 0) {  // nothing to bin: background image, empty ranges
    BinView bsz = carve_binning(nullptr, 0, f.nb, 0);
    void* bin = a->alloc_binning(a->alloc_user, bsz.bytes);
    if (bin == nullptr) return GAB200_ERR_ALLOC;
    GAB_CUDA(cudaMemsetAsync(f.g.buckets.counts, 0, f.g.bucket_clear_bytes, stream));
    const int rc = enqueue_binning_blend(f, bin, 0, 0, 0, false);
    if (rc < 0) return rc;
    st->num_rendered = st->num_candidates = 0;
    return 0;
  }

  f.ctr_host = a->counters_host;
  f.ctr_event = nullptr;
  if (mode != GAB200_SYNC_NONE) {
    if (!t_slot.ok()) return GAB200_ERR_CUDA;
    f.ctr_event = t_slot.ev;
    if (f.ctr_host == nullptr) f.ctr_host = t_slot.host;
  }
  bool bucket = a->depth_hint_hi > a->depth_hint_lo && tune_get(GAB200_TUNE_DEPTH_SORT) == 0;
  int64_t cap = speculative ? (int64_t)a->binning_hint : 0;
  int rc = enqueue_geometry(f, bucket, true, (uint32_t)cap);
  if (rc < 0) return rc;

  // the binning buffer is requested while the GPU is busy with preprocess + depth sort (in every mode)
  void* bin = nullptr;
  int64_t bin_cap = 0;
  size_t tempB = 0;
  double t_alloc = now_us();
  host_add(0, t_alloc - t0);
  if (a->binning_hint > 0) {
    bin_cap = a->binning_hint;
    tempB = f.counting ? 0 : cached_sort_temp_bytes(bin_cap, st->sort_bits);
    const BinView hv = carve_binning(nullptr, bin_cap, f.nb, tempB);
    bin = a->alloc_binning(a->alloc_user, hv.bytes);
    if (bin == nullptr) return GAB200_ERR_ALLOC;
  }
  double t1 = now_us();
  host_add(2, t1 - t_alloc);
  if (speculative) {
    rc = enqueue_binning_blend(f, bin, cap, -1, tempB, false);
    if (rc < 0) return rc;
    const double t2 = now_us();
    host_add(3, t2 - t1);
    t1 = t2;
  }
  st->depth_sort_path = bucket ? 1 : 0;
  if (mode == GAB200_SYNC_NONE) {
    st->num_rendered = st->num_candidates = -1;
    g_host_ns[5].fetch_add(1, std::memory_order_relaxed);
    return 0;
  }

  // ---- the one host wait: in the middle (EXACT) or at the end, normally already satisfied (LATE) ----
  rc = wait_counters(f);
  if (rc < 0) return rc;
  bool redo = !speculative;
  if (bucket && f.ctr_host[GAB200_CTR_BUCKET_OVERFLOW] != 0) {
    // a bucket outgrew its shared-memory budget (the hint did not fit this frame): depth order on the radix path
    bucket = false;
    st->depth_sort_path = 2;
    st->attempts++;
    rc = enqueue_geometry(f, false, false, (uint32_t)cap);
    if (rc < 0) return rc;
    rc = wait_counters(f);
    if (rc < 0) return rc;
    redo = true;
  }
  if (f.ctr_host[GAB200_CTR_NUM_RENDERED_HI] != 0) return GAB200_ERR_OVERFLOW;  // > 2^32 - 1 instances
  const int64_t N = (int64_t)f.ctr_host[GAB200_CTR_NUM_RENDERED];
  st->depth_key_min = ~f.ctr_host[GAB200_CTR_NOT_MIN_DEPTH_KEY];
  st->depth_key_max = f.ctr_host[GAB200_CTR_MAX_DEPTH_KEY];
  st->num_rendered = st->num_candidates = N;
  double t2 = now_us();
  host_add(1, t2 - t1);
  if (speculative && N > cap) {
    redo = true;
    st->attempts++;
  }
  if (redo) {
    if (bin == nullptr || N > bin_cap) {  // exact size: the layout depends on the capacity
      bin_cap = N;
      tempB = f.counting ? 0 : cached_sort_temp_bytes(bin_cap > 0 ? bin_cap : 1, st->sort_bits);
      const BinView bsz = carve_binning(nullptr, bin_cap, f.nb, tempB);
      bin = a->alloc_binning(a->alloc_user, bsz.bytes);
      if (bin == nullptr) return GAB200_ERR_ALLOC;
    }
    const double t3 = now_us();
    host_add(2, t3 - t2);
    rc = enqueue_binning_blend(f, bin, bin_cap, N, tempB, speculative);
    if (rc < 0) return rc;
    host_add(3, now_us() - t3);
  }
  g_host_ns[5].fetch_add(1, std::memory_order_relaxed);
  return N;
}

int32_t gab200_backward(const gab200_backward_args* b, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (b == nullptr || b->abi_version != GAB200_ABI_VERSION || b->fwd == nullptr || b->state == nullptr)
    return GAB200_ERR_INVALID_ARGUMENT;
  const gab200_forward_args* a = b->fwd;
  const gab200_frame_state* st = b->state;
  if (!validate(a) || !a->need_backward || b->dL_dout_color == nullptr) return GAB200_ERR_INVALID_ARGUMENT;
  if (st->geom_buffer == nullptr || st->image_buffer == nullptr || st->binning_buffer == nullptr)
    return GAB200_ERR_INVALID_ARGUMENT;
  const int P = a->P, W = a->image_width, H = a->image_height;
  const bool dbg = a->debug != 0;
  const bool bound = a->input_mode == GAB200_INPUT_BOUND_RAW;
  if (bound && a->colors_precomp == nullptr && (b->dL_dsh_dc == nullptr || (a->sh_coeffs > 1 && b->dL_dsh_rest == nullptr)))
    return GAB200_ERR_INVALID_ARGUMENT;
  if (P == 0) return GAB200_OK;
  cudaStreamCaptureStatus cap_status = cudaStreamCaptureStatusNone;
  GAB_CUDA(cudaStreamIsCapturing(stream, &cap_status));
  struct CaptureGuard {
    bool prev;
    explicit CaptureGuard(bool c) : prev(t_capturing) { t_capturing = c; }
    ~CaptureGuard() { t_capturing = prev; }
  } capture_guard(cap_status != cudaStreamCaptureStatusNone);
  GeomView g = carve_geom(st->geom_buffer, P, true, 0);
  ImageView iv = carve_image(st->image_buffer, W, H, true);
  BinView bv = carve_binning(st->binning_buffer, st->binning_capacity, true, 0);
  if (g.bytes > st->geom_bytes || iv.bytes > st->image_bytes || bv.bytes > st->binning_bytes)
    return GAB200_ERR_INVALID_ARGUMENT;  // not the buffers this forward carved

  GAB_CUDA(cudaMemsetAsync(g.g2d, 0, sizeof(float) * (size_t)P * GAB_G2D_STRIDE, stream));
  if (bound && a->binding != nullptr) {
    const size_t F = (size_t)a->num_faces;
    if (b->dL_dface_center) GAB_CUDA(cudaMemsetAsync(b->dL_dface_center, 0, sizeof(float) * 3 * F, stream));
    if (b->dL_dface_orien_mat) GAB_CUDA(cudaMemsetAsync(b->dL_dface_orien_mat, 0, sizeof(float) * 9 * F, stream));
    if (b->dL_dface_scaling) GAB_CUDA(cudaMemsetAsync(b->dL_dface_scaling, 0, sizeof(float) * F, stream));
  }
  if (b->grads_are_multicast && !bound) return GAB200_ERR_INVALID_ARGUMENT;
  if (bound && a->colors_precomp != nullptr && !b->grads_are_multicast) {
    if (b->dL_dsh_dc) GAB_CUDA(cudaMemsetAsync(b->dL_dsh_dc, 0, sizeof(float) * 3 * (size_t)P, stream));
    if (b->dL_dsh_rest && a->sh_coeffs > 1)
      GAB_CUDA(cudaMemsetAsync(b->dL_dsh_rest, 0, sizeof(float) * 3 * (size_t)(a->sh_coeffs - 1) * P, stream));
  }
  if (st->num_rendered != 0) {  // -1: only the device knows (GAB200_SYNC_NONE); empty tile lists cost nothing
    StageScope sc(GAB200_STAGE_BLEND_BWD, stream);
    launch_blend_backward(W, H, iv.ranges, iv.order, iv.order_info, bv.vals[st->sorted_selector], g.rec, a->bg, iv.final_T, iv.n_contrib,
                          b->dL_dout_color, bv.strip_mask, g.g2d, stream);
  }
  GAB_STAGE_CHECK(dbg, stream);
  {
    StageScope sc(GAB200_STAGE_PREPROCESS_BWD, stream);
    const bool csr = bound && a->binding != nullptr && b->num_face_chunks > 0 && b->face_perm && b->face_chunk_face &&
                     b->face_chunk_start && b->face_chunk_end &&
                     (b->dL_dface_center || b->dL_dface_orien_mat || b->dL_dface_scaling);
    launch_preprocess_backward(*b, g.rec, g.aux, g.clamped, g.g2d, csr ? g.face_scratch : nullptr, stream);
  }
  GAB_STAGE_CHECK(dbg, stream);
  return GAB200_OK;
}

int32_t gab200_mark_visible(int32_t P, const float* means3D, const float* viewmatrix, const float* projmatrix,
                            uint8_t* present, void* stream_) {
  (void)projmatrix;
  if (P < 0 || (P > 0 && (!means3D || !viewmatrix || !present))) return GAB200_ERR_INVALID_ARGUMENT;
  if (check_arch() < 0) return GAB200_ERR_ARCH;
  launch_mark_visible(P, means3D, viewmatrix, present, (cudaStream_t)stream_);
  return cudaPeekAtLastError() == cudaSuccess ? GAB200_OK : GAB200_ERR_CUDA;
}

int32_t gab200_bind_activate(const gab200_forward_args* a, float* means3D, float* opacities, float* scales,
                             float* cov3D, void* stream_) {
  if (a == nullptr || a->abi_version != GAB200_ABI_VERSION || a->input_mode != GAB200_INPUT_BOUND_RAW || a->P < 0)
    return GAB200_ERR_INVALID_ARGUMENT;
  if (a->P > 0 && (!a->means3D || !a->opacities || !a->scales || !a->rotations)) return GAB200_ERR_INVALID_ARGUMENT;
  if (a->binding != nullptr && (!a->face_center || !a->face_orien_mat || !a->face_scaling))
    return GAB200_ERR_INVALID_ARGUMENT;
  if (check_arch() < 0) return GAB200_ERR_ARCH;
  launch_bind_activate(*a, means3D, opacities, scales, cov3D, (cudaStream_t)stream_);
  return cudaPeekAtLastError() == cudaSuccess ? GAB200_OK : GAB200_ERR_CUDA;
}

int32_t gab200_face_frame_forward(int32_t F, int32_t V, const float* verts, const int32_t* faces, float* fc, float* fR,
                                  float* fs, void* stream_) {
  if (F < 0 || V < 0 || (F > 0 && (!verts || !faces || !fc || !fR || !fs))) return GAB200_ERR_INVALID_ARGUMENT;
  if (check_arch() < 0) return GAB200_ERR_ARCH;
  launch_face_frame_forward(F, verts, faces, fc, fR, fs, (cudaStream_t)stream_);
  return cudaPeekAtLastError() == cudaSuccess ? GAB200_OK : GAB200_ERR_CUDA;
}

int32_t gab200_face_frame_backward(int32_t F, int32_t V, const float* verts, const int32_t* faces, const float* g_fc,
                                   const float* g_fR, const float* g_fs, float* g_verts, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (F < 0 || V < 0 || (V > 0 && !g_verts) || (F > 0 && (!verts || !faces))) return GAB200_ERR_INVALID_ARGUMENT;
  if (check_arch() < 0) return GAB200_ERR_ARCH;
  GAB_CUDA(cudaMemsetAsync(g_verts, 0, sizeof(float) * 3 * (size_t)V, stream));
  launch_face_frame_backward(F, verts, faces, g_fc, g_fR, g_fs, g_verts, stream);
  return cudaPeekAtLastError() == cudaSuccess ? GAB200_OK : GAB200_ERR_CUDA;
}

static bool flame_args_ok(const gab200_flame_args* a) {
  if (a == nullptr || a->abi_version != GAB200_ABI_VERSION) return false;
  if (a->J != 5 || a->V <= 0 || a->n_shape < 0 || a->n_expr < 0 || a->T <= 0) return false;
  if (!a->v_template || !a->shapedirs || !a->posedirs || !a->J_regressor || !a->lbs_weights || !a->parents ||
      !a->J_template || !a->J_shapedirs)
    return false;
  if ((a->n_expr > 0 && !a->expr) || !a->rotation || !a->neck || !a->jaw || !a->eyes || !a->translation) return false;
  if (!a->verts || !a->workspace || ((uintptr_t)a->workspace & 255) != 0) return false;
  return true;
}

size_t gab200_flame_workspace_bytes(int32_t V, int32_t n_shape, int32_t n_expr) {
  if (V < 0 || n_shape < 0 || n_expr < 0) return 0;
  return flame_workspace_bytes(V, n_shape + n_expr);
}

int32_t gab200_flame_forward(const gab200_flame_args* a, void* stream_) {
  if (!flame_args_ok(a)) return GAB200_ERR_INVALID_ARGUMENT;
  if (check_arch() < 0) return GAB200_ERR_ARCH;
  launch_flame_forward(*a, (cudaStream_t)stream_);
  return cudaPeekAtLastError() == cudaSuccess ? GAB200_OK : GAB200_ERR_CUDA;
}

int32_t gab200_flame_backward(const gab200_flame_args* a, const float* dL_dverts, void* stream_) {
  if (!flame_args_ok(a) || dL_dverts == nullptr) return GAB200_ERR_INVALID_ARGUMENT;
  if (check_arch() < 0) return GAB200_ERR_ARCH;
  launch_flame_backward(*a, dL_dverts, (cudaStream_t)stream_);
  return cudaPeekAtLastError() == cudaSuccess ? GAB200_OK : GAB200_ERR_CUDA;
}

int32_t gab200_l1_loss_u8(int64_t n, const float* img, const uint8_t* gt, float* grad, float* loss, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (n < 0 || !loss || (n > 0 && (!img || !gt))) return GAB200_ERR_INVALID_ARGUMENT;
  if (check_arch() < 0) return GAB200_ERR_ARCH;
  GAB_CUDA(cudaMemsetAsync(loss, 0, sizeof(float), stream));
  launch_l1_loss_u8(n, img, gt, nullptr, grad, loss, stream);
  return cudaPeekAtLastError() == cudaSuccess ? GAB200_OK : GAB200_ERR_CUDA;
}

int32_t gab200_l1_loss_u8_backward(int64_t n, const float* img, const uint8_t* gt, const float* upstream, float* grad,
                                   void* stream_) {
  if (n < 0 || (n > 0 && (!img || !gt || !grad))) return GAB200_ERR_INVALID_ARGUMENT;
  if (check_arch() < 0) return GAB200_ERR_ARCH;
  launch_l1_loss_u8(n, img, gt, upstream, grad, nullptr, (cudaStream_t)stream_);
  return cudaPeekAtLastError() == cudaSuccess ? GAB200_OK : GAB200_ERR_CUDA;
}

int32_t gab200_photometric_loss(const gab200_photometric_args* a, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (a == nullptr || a->abi_version != GAB200_ABI_VERSION || a->channels < 0 || a->height < 0 || a->width < 0 ||
      a->loss == nullptr || !(a->lambda_dssim >= 0.f && a->lambda_dssim <= 1.f))
    return GAB200_ERR_INVALID_ARGUMENT;
  const int64_t n = (int64_t)a->channels * a->height * a->width;
  if (n > 0 && (!a->image || !a->gt || !a->grad || !a->scratch)) return GAB200_ERR_INVALID_ARGUMENT;
  if (check_arch() < 0) return GAB200_ERR_ARCH;
  if (n > 0 && ((uintptr_t)a->scratch & 15) != 0) return GAB200_ERR_INVALID_ARGUMENT;
  GAB_CUDA(cudaMemsetAsync(a->loss, 0, 3 * sizeof(float), stream));
  if (n > 0) GAB_CUDA(cudaMemsetAsync(a->scratch, 0, GAB_PHOTOMETRIC_SCRATCH_HEAD * sizeof(float), stream));
  launch_photometric_loss(a->channels, a->height, a->width, a->image, a->gt, a->gt_is_u8, a->lambda_dssim, a->grad,
                          a->loss, a->scratch, stream);
  return cudaPeekAtLastError() == cudaSuccess ? GAB200_OK : GAB200_ERR_CUDA;
}

int32_t gab200_adam_step(int32_t num_segments, const gab200_adam_segment* segs, int64_t step, double beta1,
                         double beta2, double eps, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (num_segments < 0 || (num_segments > 0 && segs == nullptr) || step < 1 || !(beta1 >= 0.0 && beta1 < 1.0) ||
      !(beta2 >= 0.0 && beta2 < 1.0) || !(eps >= 0.0))
    return GAB200_ERR_INVALID_ARGUMENT;
  for (int i = 0; i < num_segments; i++) {
    const gab200_adam_segment& s = segs[i];
    if (s.n < 0 || (s.n > 0 && (!s.param || !s.grad || !s.exp_avg || !s.exp_avg_sq))) return GAB200_ERR_INVALID_ARGUMENT;
  }
  if (check_arch() < 0) return GAB200_ERR_ARCH;
  launch_adam(num_segments, segs, step, beta1, beta2, eps, stream);
  return cudaPeekAtLastError() == cudaSuccess ? GAB200_OK : GAB200_ERR_CUDA;
}

int32_t gab200_nvls_allreduce(float* mc_ptr, int64_t n, int32_t rank, int32_t world, void* stream_) {
  if (mc_ptr == nullptr || n < 0 || world < 1 || rank < 0 || rank >= world || ((uintptr_t)mc_ptr & 15) != 0)
    return GAB200_ERR_INVALID_ARGUMENT;
  if (check_arch() < 0) return GAB200_ERR_ARCH;
  launch_nvls_allreduce(mc_ptr, n, rank, world, (cudaStream_t)stream_);
  return cudaPeekAtLastError() == cudaSuccess ? GAB200_OK : GAB200_ERR_CUDA;
}

static bool regularize_args_ok(const gab200_regularize_args* a, bool backward) {
  if (a == nullptr || a->abi_version != GAB200_ABI_VERSION || a->P < 0 || !a->loss || !a->sums) return false;
  if (a->P > 0 && (!a->xyz || !a->scaling || !a->radii)) return false;
  if ((a->metric_xyz || a->metric_scale) && a->binding != nullptr && !a->face_scaling) return false;
  if (backward && a->P > 0 && (!a->grad_xyz || !a->grad_scaling)) return false;
  return true;
}
int32_t gab200_regularize_forward(const gab200_regularize_args* a, void* stream_) {
  if (!regularize_args_ok(a, false)) return GAB200_ERR_INVALID_ARGUMENT;
  if (check_arch() < 0) return GAB200_ERR_ARCH;
  GAB_CUDA(launch_regularize_forward(*a, (cudaStream_t)stream_));
  return cudaPeekAtLastError() == cudaSuccess ? GAB200_OK : GAB200_ERR_CUDA;
}
int32_t gab200_regularize_backward(const gab200_regularize_args* a, const float* g_out, void* stream_) {
  if (!regularize_args_ok(a, true) || g_out == nullptr) return GAB200_ERR_INVALID_ARGUMENT;
  if (check_arch() < 0) return GAB200_ERR_ARCH;
  GAB_CUDA(launch_regularize_backward(*a, g_out, (cudaStream_t)stream_));
  return cudaPeekAtLastError() == cudaSuccess ? GAB200_OK : GAB200_ERR_CUDA;
}

size_t gab200_densify_scratch_bytes(int32_t P, int32_t F) { return densify_scratch_bytes(P < 0 ? 0 : P, F < 0 ? 0 : F); }

static bool densify_args_ok(const gab200_densify_args* a) {
  if (a == nullptr || a->abi_version != GAB200_ABI_VERSION || a->P < 0 || a->sh_rest_width < 0) return false;
  if (a->scratch == nullptr || a->totals_host == nullptr) return false;
  if (a->P > 0 && (!a->xyz || !a->rotation || !a->scaling || !a->opacity || !a->f_dc || !a->xyz_gradient_accum || !a->denom))
    return false;
  if (a->P > 0 && a->sh_rest_width > 0 && !a->f_rest) return false;
  if (a->binding != nullptr && (a->num_faces <= 0 || !a->binding_counter || !a->face_scaling)) return false;
  return true;
}

int32_t gab200_densify_plan(const gab200_densify_args* a, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (!densify_args_ok(a)) return GAB200_ERR_INVALID_ARGUMENT;
  if (check_arch() < 0) return GAB200_ERR_ARCH;
  GAB_CUDA(launch_densify_plan(*a, stream));
  GAB_CUDA(cudaStreamSynchronize(stream));  // the caller sizes the outputs from totals_host
  const uint64_t rows = (uint64_t)a->totals_host[0] + a->totals_host[1] + 2ull * a->totals_host[2];
  if (rows > 0x7fffffffull) return GAB200_ERR_OVERFLOW;
  return cudaPeekAtLastError() == cudaSuccess ? GAB200_OK : GAB200_ERR_CUDA;
}

int32_t gab200_densify_apply(const gab200_densify_args* a, const gab200_densify_out* o, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (!densify_args_ok(a) || o == nullptr || o->P_out < 0 || o->n_child_rows < 0) return GAB200_ERR_INVALID_ARGUMENT;
  if (o->P_out > 0) {
    if (!o->xyz || !o->rotation || !o->scaling || !o->opacity || !o->f_dc || !o->src_scratch || !o->kind_scratch)
      return GAB200_ERR_INVALID_ARGUMENT;
    if (a->sh_rest_width > 0 && !o->f_rest) return GAB200_ERR_INVALID_ARGUMENT;
    if (o->n_child_rows > 0 && (!o->noise || !o->noise_row_scratch)) return GAB200_ERR_INVALID_ARGUMENT;
    if (a->binding != nullptr && (!o->binding || !o->binding_counter)) return GAB200_ERR_INVALID_ARGUMENT;
  }
  if (check_arch() < 0) return GAB200_ERR_ARCH;
  GAB_CUDA(launch_densify_apply(*a, *o, stream));
  return cudaPeekAtLastError() == cudaSuccess ? GAB200_OK : GAB200_ERR_CUDA;
}

int32_t gab200_export_binning(const gab200_forward_args* a, const gab200_frame_state* st, uint64_t* keys,
                              uint32_t* values, uint32_t* ranges, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (a == nullptr || st == nullptr || st->binning_buffer == nullptr || st->image_buffer == nullptr)
    return GAB200_ERR_INVALID_ARGUMENT;
  const int W = a->image_width, H = a->image_height;
  const int gx = (W + GAB_TILE - 1) / GAB_TILE, gy = (H + GAB_TILE - 1) / GAB_TILE;
  BinView bv = carve_binning(st->binning_buffer, st->binning_capacity, a->need_backward != 0, 0);
  ImageView iv = carve_image(st->image_buffer, W, H, a->need_backward != 0);
  if (st->num_rendered < 0) return GAB200_ERR_INVALID_ARGUMENT;  // read the counters first (GAB200_SYNC_NONE)
  const size_t N = (size_t)st->num_rendered;
  if (keys && N) {
    GeomView g = carve_geom(st->geom_buffer, a->P, a->need_backward != 0, 0);
    if (st->tile_sort_path == 1)  // counting tile sort: the instance arrays hold (rank, id); the tile is in the ranges
      launch_expand_keys_by_range(gx * gy, iv.ranges, bv.vals[0], g.aux, keys, stream);
    else
      launch_expand_keys((int64_t)N, bv.keys[st->sorted_selector], bv.vals[st->sorted_selector], g.aux, keys, stream);
  }
  if (values && N) GAB_CUDA(cudaMemcpyAsync(values, bv.vals[st->sorted_selector], 4 * N, cudaMemcpyDeviceToDevice, stream));
  if (ranges) GAB_CUDA(cudaMemcpyAsync(ranges, iv.ranges, sizeof(uint2) * (size_t)gx * gy, cudaMemcpyDeviceToDevice, stream));
  return GAB200_OK;
}

}  // extern "C"
