// C ABI of the B200-native SEAM Match-RCNN retrieval hot path (see include/seam_b200.h).
// Host-side argument checking, workspace carving, tensor-map encoding and kernel launches.
// Compile: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include "../../include/seam_b200.h"
#include "aggregate_fused.cuh"
#include "backward.cuh"
#include "fold.cuh"
#include "nlb_gemm.cuh"
#include "score_exact.cuh"
#include "score_tc.cuh"
#include "tower_tc.cuh"

using namespace seam;

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct seam_handle {
  int device = 0;
  int num_sms = 0;
  float* fold = nullptr;            // folded weights (device)
  bool have_scorer = false;
  bool have_aggregator = false;
  PFN_encodeTiled encode = nullptr;
  uint64_t launches = 0;
  bool profiling = false;
  unsigned int* watchdog = nullptr;   // host-mapped record buffer of the device-side wait watchdogs
  // conv tower (f3): reorganised fp16 conv weights, biases, transposed linear weight, folded BatchNorm
  __half* tw_conv[4] = {nullptr, nullptr, nullptr, nullptr};
  float* tw_misc = nullptr;           // bias0..3 (256,256,256,1024) | lin_wt (1024*256) | lin_b | bn_scale | bn_shift
  bool have_tower = false;
  struct Span { int kernel; cudaEvent_t a, b; };
  std::vector<Span> spans;            // recorded while profiling
  std::vector<cudaEvent_t> free_events;
  char err[512] = {0};
};

// brackets one kernel launch with CUDA events on the launching stream when profiling is on
struct ProfileScope {
  seam_handle* h;
  cudaStream_t stream;
  cudaEvent_t a = nullptr, b = nullptr;
  int kernel;
  static cudaEvent_t get(seam_handle* h) {
    cudaEvent_t e = nullptr;
    if (!h->free_events.empty()) { e = h->free_events.back(); h->free_events.pop_back(); }
    else cudaEventCreate(&e);
    return e;
  }
  ProfileScope(seam_handle* h_, int kernel_, cudaStream_t s) : h(h_), stream(s), kernel(kernel_) {
    if (h->profiling && h->spans.size() < 65536) {
      a = get(h); b = get(h);
      cudaEventRecord(a, stream);
    }
  }
  ~ProfileScope() {
    if (a) {
      cudaEventRecord(b, stream);
      h->spans.push_back({kernel, a, b});
    }
  }
};

static thread_local char g_create_err[256] = "";

static unsigned int* g_watchdog_host[64] = {};

static int fail(seam_handle* h, int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  if (h) vsnprintf(h->err, sizeof(h->err), fmt, ap);
  else vsnprintf(g_create_err, sizeof(g_create_err), fmt, ap);
  va_end(ap);
  return code;
}

#define SEAM_CUDA(h, expr)                                                                             \
  do {                                                                                                 \
    cudaError_t e__ = (expr);                                                                          \
    if (e__ != cudaSuccess)                                                                            \
      return fail(h, SEAM_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, \
                  __LINE__);                                                                           \
  } while (0)

#define SEAM_LAUNCHED(h, name)                                                                      \
  do {                                                                                              \
    cudaError_t e__ = cudaGetLastError();                                                           \
    if (e__ != cudaSuccess)                                                                         \
      return fail(h, SEAM_ERR_CUDA, "launch of %s failed: %s", name, cudaGetErrorString(e__));      \
    ++(h)->launches;                                                                                \
  } while (0)

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// Full tracks / full frame blocks are fetched with one 3-D tensor-map copy: box {256, 1 track, frames} over seq viewed as
// (1+Tmax, Q, 256) with the caller's strides (elements of In: float, __half or __nv_bfloat16).  Returns whether the map
// is usable.
template <typename In>
static int encode_seq_map(seam_handle* h, const aggf::Params& p, int box_frames, CUtensorMap* tm) {
  constexpr long long ES = sizeof(In);
  memset(tm, 0, sizeof(*tm));
  if (!p.seq || p.Q <= 0 || (p.track_stride * ES) % 16 != 0 || (p.frame_stride * ES) % 16 != 0 || p.track_stride < 256 ||
      p.frame_stride < 256 || box_frames > p.Tmax)
    return 0;
  const cuuint64_t dims[3] = {256, (cuuint64_t)p.Q, (cuuint64_t)(1 + p.Tmax)};
  const cuuint64_t strides[2] = {(cuuint64_t)(p.track_stride * ES), (cuuint64_t)(p.frame_stride * ES)};
  const cuuint32_t box[3] = {256, 1, (cuuint32_t)box_frames};
  const cuuint32_t estr[3] = {1, 1, 1};
  const CUtensorMapDataType dt = std::is_same<In, __half>::value          ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16
                                 : std::is_same<In, __nv_bfloat16>::value ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                                                                          : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  return h->encode(tm, dt, 3, const_cast<void*>(p.seq), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int TR, typename In>
static void launch_aggregate_warp(seam_handle* h, aggf::Params& p, cudaStream_t stream) {
  constexpr int NW = aggf::Cfg<TR>::NW;
  const int want = (p.Q + NW - 1) / NW;
  const int grid = want < h->num_sms ? want : h->num_sms;
  CUtensorMap tm;
  p.use_tm = p.Tmax == TR ? encode_seq_map<In>(h, p, TR, &tm) : (memset(&tm, 0, sizeof(tm)), 0);
  aggf::aggregate_fused_warp_kernel<TR, In>
      <<<grid, aggf::warp_threads<TR>(), aggf::warp_smem_bytes<TR, In>(), stream>>>(tm, p);
}
template <int GW, typename In>
static void launch_aggregate_group(seam_handle* h, aggf::Params& p, cudaStream_t stream) {
  constexpr int GPC = aggf::GWARPS / GW;
  const int want = (p.Q + GPC - 1) / GPC;
  const int grid = want < h->num_sms ? want : h->num_sms;
  CUtensorMap tm;
  p.use_tm = encode_seq_map<In>(h, p, aggf::FB, &tm);
  aggf::aggregate_fused_group_kernel<GW, In><<<grid, aggf::GTHREADS, aggf::group_smem_bytes<GW, In>(), stream>>>(tm, p);
}
template <typename In>
static void launch_aggregate(seam_handle* h, aggf::Params& p, cudaStream_t stream) {
  const int Tmax = p.Tmax;
  if (Tmax <= 4) launch_aggregate_warp<4, In>(h, p, stream);
  else if (Tmax <= 10) launch_aggregate_warp<10, In>(h, p, stream);
  else if (Tmax <= 16) launch_aggregate_warp<16, In>(h, p, stream);
  else if (Tmax <= 32) launch_aggregate_group<2, In>(h, p, stream);   // two warps per track
  else launch_aggregate_group<4, In>(h, p, stream);                   // 33..64 frames: four warps per track
}
// large dynamic shared memory for the aggregation kernels of one element type
template <typename In>
static void opt_in_aggregate_smem() {
  cudaFuncSetAttribute(aggf::aggregate_fused_warp_kernel<4, In>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)aggf::warp_smem_bytes<4, In>());
  cudaFuncSetAttribute(aggf::aggregate_fused_warp_kernel<10, In>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)aggf::warp_smem_bytes<10, In>());
  cudaFuncSetAttribute(aggf::aggregate_fused_warp_kernel<16, In>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)aggf::warp_smem_bytes<16, In>());
  cudaFuncSetAttribute(aggf::aggregate_fused_group_kernel<2, In>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)aggf::group_smem_bytes<2, In>());
  cudaFuncSetAttribute(aggf::aggregate_fused_group_kernel<4, In>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)aggf::group_smem_bytes<4, In>());
}

static int import_exchange(seam_handle* h, const seam_exchange* x, xchg::Exchange* e, const char* who) {
  if (!x) return fail(h, SEAM_ERR_BAD_ARG, "%s: exchange is null", who);
  if (x->world < 1 || x->world > SEAM_MAX_WORLD || x->rank < 0 || x->rank >= x->world)
    return fail(h, SEAM_ERR_BAD_ARG, "%s: world=%d rank=%d outside [1,%d]", who, x->world, x->rank, SEAM_MAX_WORLD);
  if (x->Q < 0 || x->k < 1 || x->k > SEAM_MAX_K || x->own_max < 0)
    return fail(h, SEAM_ERR_BAD_ARG, "%s: bad Q / k / own_max", who);
  if (x->q_lo[0] != 0 || x->q_lo[x->world] != x->Q) return fail(h, SEAM_ERR_BAD_ARG, "%s: q_lo must run from 0 to Q", who);
  if (!x->step || !x->done) return fail(h, SEAM_ERR_BAD_ARG, "%s: step / done are null", who);
  memset(e, 0, sizeof(*e));
  e->world = x->world;
  e->rank = x->rank;
  e->Q = x->Q;
  e->k = x->k;
  e->own_max = x->own_max;
  const bool have_final = x->final_score[0] != nullptr;
  for (int r = 0; r <= x->world; ++r) e->q_lo[r] = x->q_lo[r];
  for (int r = 0; r < x->world; ++r) {
    if (x->q_lo[r + 1] < x->q_lo[r] || x->q_lo[r + 1] - x->q_lo[r] > x->own_max)
      return fail(h, SEAM_ERR_BAD_ARG, "%s: q_lo not monotone or ownership above own_max", who);
    if (!x->q_all[r] || !x->list_margin[r] || !x->list_idx[r] || !x->flags[r])
      return fail(h, SEAM_ERR_BAD_ARG, "%s: null buffer for rank %d", who, r);
    if (have_final && (!x->final_score[r] || !x->final_margin[r] || !x->final_idx[r]))
      return fail(h, SEAM_ERR_BAD_ARG, "%s: final buffers must be given for all ranks or none", who);
    e->q_all[r] = x->q_all[r];
    e->list_margin[r] = x->list_margin[r];
    e->list_idx[r] = x->list_idx[r];
    e->final_score[r] = have_final ? x->final_score[r] : nullptr;
    e->final_margin[r] = have_final ? x->final_margin[r] : nullptr;
    e->final_idx[r] = have_final ? x->final_idx[r] : nullptr;
    e->flags[r] = x->flags[r];
  }
  e->step = x->step;
  e->done = x->done;
  e->q_all_mc = x->world > 1 ? x->q_all_mc : nullptr;
  const bool final_mc = x->world > 1 && have_final && x->final_score_mc && x->final_margin_mc && x->final_idx_mc;
  e->final_score_mc = final_mc ? x->final_score_mc : nullptr;
  e->final_margin_mc = final_mc ? x->final_margin_mc : nullptr;
  e->final_idx_mc = final_mc ? x->final_idx_mc : nullptr;
  return SEAM_OK;
}

__global__ void device_stamp_kernel(uint64_t* dst) { *dst = ptx::globaltimer_ns(); }

extern "C" {

int seam_abi_version(void) { return 3; }

size_t seam_exchange_sizeof(void) { return sizeof(seam_exchange); }

int seam_create(seam_handle** out, int device) {
  if (!out) return fail(nullptr, SEAM_ERR_BAD_ARG, "seam_create: out is null");
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(nullptr, SEAM_ERR_CUDA, "no CUDA device available (%s); this library has no CPU path",
                e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
  if (device < 0 || device >= ndev) return fail(nullptr, SEAM_ERR_BAD_ARG, "device %d out of range", device);
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess)
    return fail(nullptr, SEAM_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
  if (prop.major != 10)
    return fail(nullptr, SEAM_ERR_UNSUPPORTED, "device %d is sm_%d%d; this library is built for sm_100a only", device,
                prop.major, prop.minor);
  seam_handle* h = new (std::nothrow) seam_handle();
  if (!h) return fail(nullptr, SEAM_ERR_CUDA, "out of host memory");
  h->device = device;
  h->num_sms = prop.multiProcessorCount;
  DeviceGuard guard(device);
  if ((e = cudaMalloc(&h->fold, sizeof(float) * Fold::TOTAL)) != cudaSuccess) {
    delete h;
    return fail(nullptr, SEAM_ERR_CUDA, "cudaMalloc(fold): %s", cudaGetErrorString(e));
  }
  cudaMemset(h->fold, 0, sizeof(float) * Fold::TOTAL);
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) {
    cudaFree(h->fold);
    delete h;
    return fail(nullptr, SEAM_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
  }
  h->encode = reinterpret_cast<PFN_encodeTiled>(fn);
  // watchdog records live in host-mapped memory so that they survive a trapped launch: one buffer per
  // device for the life of the process (the device-side pointer must never dangle)
  if (device < 64) {
    if (!g_watchdog_host[device]) {
      unsigned int* hp = nullptr;
      if (cudaHostAlloc(reinterpret_cast<void**>(&hp), 1024, cudaHostAllocMapped) == cudaSuccess) {
        memset(hp, 0, 1024);
        unsigned int* dptr = nullptr;
        if (cudaHostGetDevicePointer(reinterpret_cast<void**>(&dptr), hp, 0) == cudaSuccess &&
            cudaMemcpyToSymbol(ptx::g_watchdog, &dptr, sizeof(dptr)) == cudaSuccess)
          g_watchdog_host[device] = hp;
      }
      cudaGetLastError();
    }
    h->watchdog = g_watchdog_host[device];
  }
  // opt in to large dynamic shared memory once
  cudaFuncSetAttribute(score::score_topk_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)score::SMEM_BYTES);
  cudaFuncSetAttribute(score::score_topk_kernel<score::VAR_RANK>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)score::SMEM_BYTES);
  opt_in_aggregate_smem<float>();
  opt_in_aggregate_smem<__half>();
  opt_in_aggregate_smem<__nv_bfloat16>();
  cudaFuncSetAttribute(bwd::agg_backward_folded_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)bwd::agg_bwd_smem_bytes(SEAM_MAX_T));
  cudaFuncSetAttribute(tower::conv3x3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tower::SMEM_BYTES);
  cudaFuncSetAttribute(nlbgemm::nlb_full_front_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)((SEAM_MAX_T * 257 + 2 * SEAM_MAX_T) * sizeof(float)));
  if ((e = cudaGetLastError()) != cudaSuccess) {
    cudaFree(h->fold);
    delete h;
    return fail(nullptr, SEAM_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  }
  *out = h;
  return SEAM_OK;
}

void seam_destroy(seam_handle* h) {
  if (!h) return;
  {
    DeviceGuard guard(h->device);
    for (auto& sp : h->spans) { cudaEventDestroy(sp.a); cudaEventDestroy(sp.b); }
    for (auto e : h->free_events) cudaEventDestroy(e);
    cudaFree(h->fold);
    for (int i = 0; i < 4; ++i) cudaFree(h->tw_conv[i]);
    cudaFree(h->tw_misc);
  }
  delete h;
}

int seam_watchdog_read(const seam_handle* h, uint32_t* out, int max_records) {
  if (!h || !h->watchdog || !out || max_records <= 0) return 0;
  const volatile unsigned int* w = h->watchdog;
  int n = (int)w[0];
  if (n > ptx::WATCHDOG_RECORDS) n = ptx::WATCHDOG_RECORDS;
  if (n > max_records) n = max_records;
  for (int i = 0; i < n * 8; ++i) out[i] = w[8 + i];
  return n;
}

int seam_device_stamp(seam_handle* h, uint64_t* dst, void* stream) {
  if (!h || !dst) return SEAM_ERR_BAD_ARG;
  DeviceGuard guard(h->device);
  device_stamp_kernel<<<1, 1, 0, static_cast<cudaStream_t>(stream)>>>(dst);
  return SEAM_OK;
}

const char* seam_last_error(const seam_handle* h) { return h ? h->err : g_create_err; }

uint64_t seam_launch_count(const seam_handle* h) { return h ? h->launches : 0; }

int seam_profile_enable(seam_handle* h, int enable) {
  if (!h) return SEAM_ERR_BAD_ARG;
  h->profiling = enable != 0;
  return SEAM_OK;
}

int seam_profile_read(seam_handle* h, int kernel, double* total_ms, int* launches) {
  if (!h || !total_ms || !launches) return SEAM_ERR_BAD_ARG;
  DeviceGuard guard(h->device);
  double tot = 0.0;
  int n = 0;
  std::vector<seam_handle::Span> keep;
  for (auto& sp : h->spans) {
    if (sp.kernel != kernel) { keep.push_back(sp); continue; }
    SEAM_CUDA(h, cudaEventSynchronize(sp.b));
    float ms = 0.f;
    SEAM_CUDA(h, cudaEventElapsedTime(&ms, sp.a, sp.b));
    tot += ms;
    ++n;
    h->free_events.push_back(sp.a);
    h->free_events.push_back(sp.b);
  }
  h->spans.swap(keep);
  *total_ms = tot;
  *launches = n;
  return SEAM_OK;
}

int seam_load_weights(seam_handle* h, const seam_weights* w, void* stream_) {
  if (!h) return SEAM_ERR_BAD_ARG;
  if (!w) return fail(h, SEAM_ERR_BAD_ARG, "seam_load_weights: weights struct is null");
  const float* const* ptrs = reinterpret_cast<const float* const*>(w);
  for (int i = 0; i < 13; ++i)
    if (!ptrs[i]) return fail(h, SEAM_ERR_BAD_ARG, "seam_load_weights: weight pointer %d is null", i);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  FoldIn in{w->theta_w, w->theta_b, w->phi_w, w->phi_b, w->g_w,    w->g_b,   w->W_w,
            w->W_b,     w->concat_w, w->att_w, w->att_b, w->last_w, w->last_b};
  fold_vectors_kernel<<<1, 256, 0, stream>>>(in, h->fold);
  SEAM_LAUNCHED(h, "fold_vectors_kernel");
  fold_matrix_kernel<<<256, 256, 0, stream>>>(w->W_w, w->g_w, h->fold);
  SEAM_LAUNCHED(h, "fold_matrix_kernel");
  fold_m16_kernel<<<256, 256, 0, stream>>>(h->fold);
  SEAM_LAUNCHED(h, "fold_m16_kernel");
  h->have_scorer = h->have_aggregator = true;
  return SEAM_OK;
}

int seam_load_scorer(seam_handle* h, const float* last_w, const float* last_b, void* stream_) {
  if (!h) return SEAM_ERR_BAD_ARG;
  if (!last_w || !last_b) return fail(h, SEAM_ERR_BAD_ARG, "seam_load_scorer: null pointer");
  DeviceGuard guard(h->device);
  fold_scorer_kernel<<<1, 256, 0, static_cast<cudaStream_t>(stream_)>>>(last_w, last_b, h->fold);
  SEAM_LAUNCHED(h, "fold_scorer_kernel");
  h->have_scorer = true;
  return SEAM_OK;
}

// ------------------------------------------------------------------------------ aggregation
size_t seam_aggregate_workspace_bytes(int Q) {
  (void)Q;
  return 256;   // the fused kernel keeps every intermediate on the SM
}

// the element type of a track tensor x3_1_seq, as the entry point that received it says
enum class TrackType { F32, F16, BF16 };

// seq holds values of type tt (strides in elements)
static int aggregate_impl(seam_handle* h, const xchg::Exchange* x, int row0, int last, const void* seq, TrackType tt,
                          const uint8_t* mask, const int32_t* lens, int Tmax, int Q, int64_t frame_stride,
                          int64_t track_stride, float* out, float* att, cudaStream_t stream, const char* who) {
  if (!h->have_aggregator) return fail(h, SEAM_ERR_STATE, "%s: weights not loaded", who);
  if (Q < 0 || Tmax < 0) return fail(h, SEAM_ERR_BAD_ARG, "%s: negative size", who);
  if (!x && Q == 0) return SEAM_OK;
  if (!x && !out) return fail(h, SEAM_ERR_BAD_ARG, "%s: out is null", who);
  if (Tmax > SEAM_MAX_T) return fail(h, SEAM_ERR_UNSUPPORTED, "%s: Tmax=%d exceeds %d", who, Tmax, SEAM_MAX_T);
  DeviceGuard guard(h->device);
  if (!x && Tmax == 0) {   // only the dummy row: every track is empty -> zero descriptors
    SEAM_CUDA(h, cudaMemsetAsync(out, 0, (size_t)Q * 256 * 4, stream));
    return SEAM_OK;
  }
  if (Q > 0 && Tmax > 0 && !seq) return fail(h, SEAM_ERR_BAD_ARG, "%s: null pointer", who);
  // the bulk copies and the tensor map move whole frames: 16-byte aligned rows
  const int64_t stride_mask = tt == TrackType::F32 ? 3 : 7;
  if (!aligned16(seq) || (out && !aligned16(out)) || (frame_stride & stride_mask) || (track_stride & stride_mask))
    return fail(h, SEAM_ERR_UNSUPPORTED, "%s: seq/out must be 16-byte aligned, strides multiples of %s", who,
                tt == TrackType::F32 ? "4" : tt == TrackType::F16 ? "8 fp16 elements" : "8 bf16 elements");
  ProfileScope prof(h, SEAM_KERNEL_AGGREGATE, stream);
  aggf::Params p;
  memset(&p, 0, sizeof(p));
  p.seq = seq;
  p.mask = mask;
  p.lens = lens;
  p.Tmax = Tmax;
  p.Q = Q;
  p.frame_stride = frame_stride;
  p.track_stride = track_stride;
  p.fold = h->fold;
  p.out = out;
  p.att = att;
  if (x) {
    p.x_on = 1;
    p.x_last = last;
    p.x_row0 = row0;
    p.x = *x;
    // a rank without tracks in this call (or with empty tracks only: Tmax == 0) still has to take part in the
    // protocol: one CTA, zero tracks / zero-length tracks, descriptors = 0
    if (Tmax == 0) { p.Tmax = 1; p.lens = nullptr; p.mask = nullptr; p.seq = nullptr; p.Q = -Q; }
  }
  if (p.Q < 0) return fail(h, SEAM_ERR_UNSUPPORTED, "%s: Tmax == 0 in the sharded search", who);
  if (p.Q == 0) {
    // nothing to aggregate on this rank: only the signal is needed
    if (x && last) {
      aggf::signal_only_kernel<<<1, 32, 0, stream>>>(p.x);
      SEAM_LAUNCHED(h, "signal_only_kernel");
    }
    return SEAM_OK;
  }
  if (tt == TrackType::F16) launch_aggregate<__half>(h, p, stream);
  else if (tt == TrackType::BF16) launch_aggregate<__nv_bfloat16>(h, p, stream);
  else launch_aggregate<float>(h, p, stream);
  SEAM_LAUNCHED(h, "aggregate kernel");
  return SEAM_OK;
}

int seam_aggregate(seam_handle* h, const float* seq, const uint8_t* mask, const int32_t* lens, int Tmax, int Q,
                   int64_t frame_stride, int64_t track_stride, float* out, float* att, void* workspace,
                   size_t workspace_bytes, void* stream_) {
  (void)workspace;
  (void)workspace_bytes;
  if (!h) return SEAM_ERR_BAD_ARG;
  return aggregate_impl(h, nullptr, 0, 0, seq, TrackType::F32, mask, lens, Tmax, Q, frame_stride, track_stride, out,
                        att, static_cast<cudaStream_t>(stream_), "seam_aggregate");
}

int seam_aggregate_f16(seam_handle* h, const void* seq, const uint8_t* mask, const int32_t* lens, int Tmax, int Q,
                       int64_t frame_stride, int64_t track_stride, float* out, float* att, void* workspace,
                       size_t workspace_bytes, void* stream_) {
  (void)workspace;
  (void)workspace_bytes;
  if (!h) return SEAM_ERR_BAD_ARG;
  return aggregate_impl(h, nullptr, 0, 0, seq, TrackType::F16, mask, lens, Tmax, Q, frame_stride, track_stride, out,
                        att, static_cast<cudaStream_t>(stream_), "seam_aggregate_f16");
}

int seam_aggregate_bf16(seam_handle* h, const void* seq, const uint8_t* mask, const int32_t* lens, int Tmax, int Q,
                        int64_t frame_stride, int64_t track_stride, float* out, float* att, void* workspace,
                        size_t workspace_bytes, void* stream_) {
  (void)workspace;
  (void)workspace_bytes;
  if (!h) return SEAM_ERR_BAD_ARG;
  return aggregate_impl(h, nullptr, 0, 0, seq, TrackType::BF16, mask, lens, Tmax, Q, frame_stride, track_stride, out,
                        att, static_cast<cudaStream_t>(stream_), "seam_aggregate_bf16");
}

static int sharded_aggregate_impl(seam_handle* h, const seam_exchange* x, const void* seq, TrackType tt,
                                  const uint8_t* mask, const int32_t* lens, int Tmax, int Qlocal, int64_t frame_stride,
                                  int64_t track_stride, int row0, int last, float* att, void* stream_, const char* who) {
  if (!h) return SEAM_ERR_BAD_ARG;
  xchg::Exchange e;
  int rc = import_exchange(h, x, &e, who);
  if (rc != SEAM_OK) return rc;
  if (row0 < 0 || Qlocal < 0 || row0 + Qlocal > x->Q)
    return fail(h, SEAM_ERR_BAD_ARG, "%s: rows [%d,%d) outside the %d queries", who, row0, row0 + Qlocal, x->Q);
  return aggregate_impl(h, &e, row0, last ? 1 : 0, seq, tt, mask, lens, Tmax, Qlocal, frame_stride, track_stride,
                        nullptr, att, static_cast<cudaStream_t>(stream_), who);
}

int seam_sharded_aggregate(seam_handle* h, const seam_exchange* x, const float* seq, const uint8_t* mask,
                           const int32_t* lens, int Tmax, int Qlocal, int64_t frame_stride, int64_t track_stride,
                           int row0, int last, float* att, void* stream_) {
  return sharded_aggregate_impl(h, x, seq, TrackType::F32, mask, lens, Tmax, Qlocal, frame_stride, track_stride, row0,
                                last, att, stream_, "seam_sharded_aggregate");
}

int seam_sharded_aggregate_f16(seam_handle* h, const seam_exchange* x, const void* seq, const uint8_t* mask,
                               const int32_t* lens, int Tmax, int Qlocal, int64_t frame_stride, int64_t track_stride,
                               int row0, int last, float* att, void* stream_) {
  return sharded_aggregate_impl(h, x, seq, TrackType::F16, mask, lens, Tmax, Qlocal, frame_stride, track_stride, row0,
                                last, att, stream_, "seam_sharded_aggregate_f16");
}

int seam_sharded_aggregate_bf16(seam_handle* h, const seam_exchange* x, const void* seq, const uint8_t* mask,
                                const int32_t* lens, int Tmax, int Qlocal, int64_t frame_stride, int64_t track_stride,
                                int row0, int last, float* att, void* stream_) {
  return sharded_aggregate_impl(h, x, seq, TrackType::BF16, mask, lens, Tmax, Qlocal, frame_stride, track_stride, row0,
                                last, att, stream_, "seam_sharded_aggregate_bf16");
}

size_t seam_nlb_workspace_bytes(int B, int T) {
  if (B <= 0 || T <= 0) return 256;
  const size_t rows = (size_t)B * T;
  return 2 * align_up(rows * 256 * 4, 256) + align_up(rows * 2 * 4, 256);
}

int seam_nlb_forward(seam_handle* h, const float* x, int B, int T, float* z, void* workspace, size_t workspace_bytes,
                     void* stream_) {
  if (!h) return SEAM_ERR_BAD_ARG;
  if (!h->have_aggregator) return fail(h, SEAM_ERR_STATE, "seam_nlb_forward: weights not loaded");
  if (B < 0 || T < 0) return fail(h, SEAM_ERR_BAD_ARG, "seam_nlb_forward: negative size");
  if (B == 0 || T == 0) return SEAM_OK;
  if (T > SEAM_MAX_T) return fail(h, SEAM_ERR_UNSUPPORTED, "seam_nlb_forward: T=%d exceeds %d", T, SEAM_MAX_T);
  if (!x || !z || !workspace) return fail(h, SEAM_ERR_BAD_ARG, "seam_nlb_forward: null pointer");
  if (workspace_bytes < seam_nlb_workspace_bytes(B, T))
    return fail(h, SEAM_ERR_STATE, "seam_nlb_forward: workspace too small");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  const size_t rows = (size_t)B * T;
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  float* Xt = reinterpret_cast<float*>(ws);
  float* R = reinterpret_cast<float*>(ws + align_up(rows * 256 * 4, 256));
  float* sv = reinterpret_cast<float*>(ws + 2 * align_up(rows * 256 * 4, 256));
  const size_t smem = (size_t)(T * 257 + 2 * T) * sizeof(float);
  nlbgemm::nlb_full_front_kernel<<<B, 256, smem, stream>>>(x, T, h->fold, Xt, R, sv);
  SEAM_LAUNCHED(h, "nlb_full_front_kernel");
  nlbgemm::Params gp;
  gp.pooled = Xt;
  gp.R = R;
  gp.sv = sv;
  gp.fold = h->fold;
  gp.out = z;
  gp.rows = (int)rows;
  gp.T = T;
  dim3 ggrid((unsigned)((rows + nlbgemm::TM - 1) / nlbgemm::TM), 256 / nlbgemm::TN);
  {
    ProfileScope prof(h, SEAM_KERNEL_NLB_GEMM, stream);
    nlbgemm::nlb_gemm_simt_kernel<<<ggrid, 256, 0, stream>>>(gp);
    SEAM_LAUNCHED(h, "nlb_gemm_simt_kernel");
  }
  return SEAM_OK;
}

// ------------------------------------------------------------------------------ scorer
// the element type of a gallery's (G,256) rows, as the entry point that received them says.  An fp16 gallery is its own
// tensor-core operand (g16 is the same pointer as the rows); fp32 and bf16 rows have a separate fp16 image g16.
enum class RowType { F32, F16, BF16 };

// rows: the gallery's (G,256) rows of type rt.  For an fp16 gallery g16 is the same pointer and is not written.
static int prepare_gallery_impl(seam_handle* h, const void* rows, RowType rt, void* g16, int G, float* cg,
                                float* gstat, void* stream_, const char* who) {
  if (!h) return SEAM_ERR_BAD_ARG;
  if (!h->have_scorer) return fail(h, SEAM_ERR_STATE, "%s: scorer weights not loaded", who);
  if (G < 0) return fail(h, SEAM_ERR_BAD_ARG, "%s: negative size", who);
  if (!gstat) return fail(h, SEAM_ERR_BAD_ARG, "%s: gstat is null", who);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  SEAM_CUDA(h, cudaMemsetAsync(gstat, 0, 16, stream));
  if (G == 0) return SEAM_OK;
  if (!rows || !g16 || !cg) return fail(h, SEAM_ERR_BAD_ARG, "%s: null pointer", who);
  if (!aligned16(rows) || !aligned16(g16)) return fail(h, SEAM_ERR_UNSUPPORTED, "%s: 16-byte alignment", who);
  {
    ProfileScope prof(h, SEAM_KERNEL_PREP_GALLERY, stream);
    if (rt == RowType::F16)
      exact::prep_gallery_kernel<__half><<<(G + 7) / 8, 256, 0, stream>>>(static_cast<const __half*>(rows), G, h->fold,
                                                                          nullptr, cg, gstat);
    else if (rt == RowType::BF16)
      exact::prep_gallery_kernel<__nv_bfloat16><<<(G + 7) / 8, 256, 0, stream>>>(
          static_cast<const __nv_bfloat16*>(rows), G, h->fold, static_cast<__half*>(g16), cg, gstat);
    else
      exact::prep_gallery_kernel<float><<<(G + 7) / 8, 256, 0, stream>>>(static_cast<const float*>(rows), G, h->fold,
                                                                         static_cast<__half*>(g16), cg, gstat);
    SEAM_LAUNCHED(h, "prep_gallery_kernel");
  }
  return SEAM_OK;
}

int seam_prepare_gallery(seam_handle* h, const float* g, int G, void* g16, float* cg, float* gstat, void* stream_) {
  return prepare_gallery_impl(h, g, RowType::F32, g16, G, cg, gstat, stream_, "seam_prepare_gallery");
}

int seam_prepare_gallery_f16(seam_handle* h, const void* g16, int G, float* cg, float* gstat, void* stream_) {
  return prepare_gallery_impl(h, g16, RowType::F16, const_cast<void*>(g16), G, cg, gstat, stream_,
                              "seam_prepare_gallery_f16");
}

int seam_prepare_gallery_bf16(seam_handle* h, const void* g, int G, void* g16, float* cg, float* gstat, void* stream_) {
  return prepare_gallery_impl(h, g, RowType::BF16, g16, G, cg, gstat, stream_, "seam_prepare_gallery_bf16");
}

struct ScorePlan {
  int num_mtiles, P, CAP, nseed;
  score::TilePlan tiles;
  size_t xunits;   // the exhaustive kernel's partial-list units (off_xpart)
  size_t off_a16, off_rq, off_anorm, off_thr, off_rowcnt, off_gmax, off_rowflag, off_rowbuf, off_cnt, off_rows, off_xpart, off_xdone, total;
};

// The (query tile, gallery tile) grid is linearised query-major and cut into one contiguous
// range per CTA (score_tc.cuh).  A query tile's gallery sweep is therefore shared by at most P
// CTAs ("pieces"); each piece owns 4 candidate sub-lists per row (one per epilogue thread of
// the row) of CAP entries, CAP >= 3 times the expected number of appends.
static ScorePlan plan_score(int num_sms, int Q, int G, bool rank) {
  ScorePlan s;
  score::TilePlan& tp = s.tiles;
  s.num_mtiles = (Q + score::BM - 1) / score::BM;
  tp.ntiles_n = (G + score::BN - 1) / score::BN;
  if (s.num_mtiles < 1) s.num_mtiles = 1;
  if (tp.ntiles_n < 1) tp.ntiles_n = 1;
  const long long ntn = tp.ntiles_n, total = (long long)s.num_mtiles * ntn;
  tp.nb = total < num_sms ? (int)total : num_sms;
  if (tp.nb > score::MAX_GRID) tp.nb = score::MAX_GRID;
  const int grid = tp.nb;
  int* tb = tp.tb;
  s.nseed = rank ? 0 : score::NSEED;
  // Cost-balanced contiguous ranges.  A tile costs 1; a segment start costs SEG_COST (query tile load,
  // epilogue hand-over); a segment that holds its row's first gallery tile -- or is all a CTA has --
  // also sweeps min(nseed, length) threshold-only sample tiles (score_tc.cuh, segment_before).  walk()
  // cuts ranges of cost <= target; the smallest target whose last range also fits is found by bisection.
  const double SEG_COST = 0.35;
  auto walk = [&](double target) -> double {   // returns the cost of the last CTA's range
    long long pos = 0;
    tb[0] = 0;
    for (int b = 0; b < grid; ++b) {
      const long long t0 = pos;
      double cost = 0.0;
      const bool last = b == grid - 1;
      while (pos < total) {
        const long long row_end = (pos / ntn + 1) * ntn;
        const long long seg_len = row_end - pos;
        const bool head = pos % ntn == 0;
        const double samples = (double)(seg_len < s.nseed ? seg_len : s.nseed);
        double over = SEG_COST + (head ? samples : 0.0);
        // the tail of a row that leaves no room for the next row's head is all this CTA sweeps: sampled
        if (!head && pos == t0 && (double)seg_len + over + SEG_COST + s.nseed + 1.0 > target) over += samples;
        long long n = seg_len;
        if (!last) {
          const double room = target - cost - over;
          if (room < 1.0 && pos > t0) break;             // not worth starting another segment
          const long long fit = room < 1.0 ? 1 : (long long)room;
          if (fit < n) n = fit;
        }
        cost += over + (double)n;
        pos += n;
        if (pos < row_end) break;                        // budget exhausted inside the row
      }
      tb[b + 1] = (int)pos;
      if (last) return cost;
    }
    return 0.0;
  };
  {
    // every query tile starts a segment, every CTA boundary at most one more
    const double all = (double)total + ((double)s.num_mtiles + grid) * (SEG_COST + s.nseed);
    double lo = (double)total / grid, hi = 2.0 * all / grid + s.nseed + 2.0;
    for (int it = 0; it < 40; ++it) {
      const double mid = 0.5 * (lo + hi);
      if (walk(mid) <= mid) hi = mid;
      else lo = mid;
    }
    walk(hi);
    tb[grid] = (int)total;
  }
  // sub-list slots per row = most CTAs whose ranges touch one query tile's sweep (pieces are numbered
  // from the first CTA that touches the row)
  int pmax = 1;
  long long max_range = 1;
  {
    int b_first = 0;
    for (long long m = 0; m < s.num_mtiles; ++m) {
      const long long r0 = m * ntn, r1 = r0 + ntn;
      while (b_first + 1 < grid && tb[b_first + 1] <= r0) ++b_first;   // first CTA with tb[b+1] > r0
      int b_last = b_first;
      while (b_last + 1 < grid && tb[b_last + 1] < r1) ++b_last;
      if (b_last - b_first + 1 > pmax) pmax = b_last - b_first + 1;
    }
    for (int b = 0; b < grid; ++b)
      if (tb[b + 1] - tb[b] > max_range) max_range = tb[b + 1] - tb[b];
  }
  s.P = pmax;
  // Expected bytes one epilogue thread appends over a piece of T tiles.  A record is a quad of 4 adjacent
  // columns (16 bytes), appended when its maximum beats the row's bound: with a cold bound a whole tile
  // (16 quads) goes out, later about 32/t items per tile t (about 130 items sit above a row's 32-group
  // bound, a quarter of them in this thread's columns), nearly all in different quads; seeded pieces start
  // at the rate of tile nseed+1.  Segments shorter than 4*nseed tiles run unseeded and may append whole
  // tiles.  3x margin on the sparse part.
  const double T = (double)(max_range < ntn ? max_range : ntn);
  const double tile_bytes = score::QCOLS / 4 * 16.0;
  double need;
  if (s.nseed > 0) {
    const double short_tiles = T < 4.0 * s.nseed - 1.0 ? T : 4.0 * s.nseed - 1.0;
    need = short_tiles * tile_bytes;
    if (T >= 4.0 * s.nseed) {
      const double seeded = 16.0 * 3.0 * (16.0 + 32.0 * log((T + s.nseed) / s.nseed));
      if (seeded > need) need = seeded;
    }
  } else {
    need = 16.0 * 3.0 * (64.0 + 32.0 * log(T));
  }
  if (need > T * tile_bytes) need = T * tile_bytes;          // a thread cannot append more than it sees
  if (rank) {
    // rank-of-target variant: a thread appends the quads holding an element inside the band around the
    // target's value -- about 1-2 % of its columns for a target in the bulk of the ranking; budget 6 %
    const double band = 0.06 * T * score::QCOLS * 16.0;
    if (band > need) need = band;
  }
  need += tile_bytes;                                        // a list closes one tile before it is full
  int cap = 2 * score::QCOLS;                                // 8-byte units; power of two: a sub-list is aligned to its size
  while (cap * 8 < (int)need && cap < 8192) cap *= 2;
  s.CAP = cap;
  const size_t nlists = (size_t)s.P * score::NQ;
  size_t o = 0;
  s.off_a16 = o;     o += align_up((size_t)Q * 256 * 2, 256);
  s.off_rq = o;      o += align_up((size_t)Q * 4, 256);
  s.off_anorm = o;   o += align_up((size_t)Q * 4, 256);
  s.off_thr = o;     o += align_up((size_t)Q * 4, 256);
  s.off_rowcnt = o;  o += align_up((size_t)Q * nlists * 4, 256);
  s.off_gmax = o;    o += align_up((size_t)Q * nlists * score::GROUPS * 4, 256);
  s.off_rowflag = o; o += align_up((size_t)Q * 4, 256);
  s.off_rowbuf = o;  o += align_up((size_t)Q * nlists * s.CAP * 8 + (size_t)s.CAP * 8, 256);   // + slack to align the base
  s.off_cnt = o;     o += 256;
  s.off_rows = o;    o += align_up((size_t)Q * 4, 256);
  // exhaustive kernel: per-slice lists of rows split over several CTAs (units <= max(its grid, Q)), per-row counts
  s.xunits = (size_t)(Q > 2 * num_sms ? Q : 2 * num_sms);
  s.off_xpart = o;   o += align_up(s.xunits * 32 * 8, 256);
  s.off_xdone = o;   o += align_up((size_t)Q * 4, 256);
  s.total = o;
  return s;
}

size_t seam_score_workspace_bytes(const seam_handle* h, int Q, int G, int k) {
  (void)k;
  if (!h || Q <= 0 || G <= 0) return 256;
  return plan_score(h->num_sms, Q, G, false).total;
}

int seam_score_plan(const seam_handle* h, int Q, int G, int64_t* out) {
  if (!h || !out || Q <= 0 || G <= 0) return SEAM_ERR_BAD_ARG;
  const ScorePlan s = plan_score(h->num_sms, Q, G, false);
  const int64_t v[14] = {s.num_mtiles, s.tiles.ntiles_n, s.tiles.nb, s.P, s.CAP, (int64_t)s.off_a16,
                         (int64_t)s.off_rq, (int64_t)s.off_anorm, (int64_t)s.off_thr, (int64_t)s.off_rowcnt,
                         (int64_t)s.off_rowbuf, (int64_t)s.off_cnt, (int64_t)s.off_rows, (int64_t)s.total};
  for (int i = 0; i < 14; ++i) out[i] = v[i];
  return SEAM_OK;
}

// Pure host logic (no handle, no device): the tile ranges of the scorer's persistent CTAs.
int seam_score_partition(int num_sms, int Q, int G, int rank_variant, int32_t* bounds, int bounds_len, int32_t* out6) {
  if (num_sms < 1 || Q <= 0 || G <= 0 || !bounds || !out6) return SEAM_ERR_BAD_ARG;
  const ScorePlan s = plan_score(num_sms, Q, G, rank_variant != 0);
  if (bounds_len < s.tiles.nb + 1) return SEAM_ERR_BAD_ARG;
  for (int b = 0; b <= s.tiles.nb; ++b) bounds[b] = s.tiles.tb[b];
  out6[0] = s.num_mtiles;
  out6[1] = s.tiles.ntiles_n;
  out6[2] = s.tiles.nb;
  out6[3] = s.P;
  out6[4] = s.CAP;
  out6[5] = s.nseed;
  return SEAM_OK;
}

__global__ void fill_empty_topk_kernel(float* s, float* d, int32_t* i, size_t n) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) {
    s[t] = 0.f;
    d[t] = -INFINITY;
    i[t] = -1;
  }
}

static int encode_map_fp16_rows(seam_handle* h, CUtensorMap* map, const void* base, int rows, int box_rows) {
  const cuuint64_t dims[2] = {256, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {256 * 2};
  const cuuint32_t box[2] = {(cuuint32_t)score::BK, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = h->encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(h, SEAM_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return SEAM_OK;
}

// The scorer's workspace, carved by plan_score's offsets into typed buffers.
struct ScoreWorkspace {
  ScorePlan plan;
  __half* a16;
  float *rq, *anorm, *gmax;
  uint32_t *thr, *rowcnt, *rowflag;
  uint2* rowbuf;
  int32_t *counters, *frows;
  float* xpart_d;              // exhaustive kernel
  int32_t *xpart_i, *xdone;
  // rank variant only (null otherwise): it keeps no group maxima, and its per-sub-list counts of the elements
  // above the band (Q x nlists), the band (lo, hi] and the target margins (Q each) live in that region
  int32_t* above;
  float *lo, *hi, *dtarget;
};

// Checks what both scorer variants take, plans the work and carves the workspace; fn names the entry point, rows are
// the gallery rows the direct form reads (g, or g16 itself for an fp16 gallery).
static int carve_score_workspace(seam_handle* h, const char* fn, bool rank, const float* q, int Q, const void* rows,
                                 const void* g16, const float* cg, const float* gstat, int G, void* workspace,
                                 size_t workspace_bytes, ScoreWorkspace* w) {
  if (!q || !rows || !g16 || !cg || !gstat || !workspace) return fail(h, SEAM_ERR_BAD_ARG, "%s: null pointer", fn);
  if (!aligned16(q) || !aligned16(rows) || !aligned16(g16) || (reinterpret_cast<uintptr_t>(workspace) & 255u))
    return fail(h, SEAM_ERR_UNSUPPORTED, "%s: q/g/g16 need 16-byte, workspace 256-byte alignment", fn);
  const ScorePlan& s = w->plan = plan_score(h->num_sms, Q, G, rank);
  if (s.tiles.ntiles_n > score::TAG_TILES)
    return fail(h, SEAM_ERR_UNSUPPORTED, "%s: G=%d exceeds the %d gallery rows one shard may hold", fn, G,
                score::TAG_TILES * score::BN);
  if (workspace_bytes < s.total)
    return fail(h, SEAM_ERR_STATE, "%s: workspace too small (%zu < %zu)", fn, workspace_bytes, s.total);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  w->a16 = reinterpret_cast<__half*>(ws + s.off_a16);
  w->rq = reinterpret_cast<float*>(ws + s.off_rq);
  w->anorm = reinterpret_cast<float*>(ws + s.off_anorm);
  w->thr = reinterpret_cast<uint32_t*>(ws + s.off_thr);
  w->rowcnt = reinterpret_cast<uint32_t*>(ws + s.off_rowcnt);
  w->gmax = reinterpret_cast<float*>(ws + s.off_gmax);
  w->rowflag = reinterpret_cast<uint32_t*>(ws + s.off_rowflag);
  // sub-lists are aligned to their (power-of-two) size so that none straddles a 4 GiB boundary
  w->rowbuf = reinterpret_cast<uint2*>(align_up(reinterpret_cast<uintptr_t>(ws + s.off_rowbuf), (size_t)s.CAP * 8));
  w->counters = reinterpret_cast<int32_t*>(ws + s.off_cnt);
  w->frows = reinterpret_cast<int32_t*>(ws + s.off_rows);
  w->xpart_d = reinterpret_cast<float*>(ws + s.off_xpart);
  w->xpart_i = reinterpret_cast<int32_t*>(ws + s.off_xpart + s.xunits * 32 * 4);
  w->xdone = reinterpret_cast<int32_t*>(ws + s.off_xdone);
  const size_t nlists = (size_t)s.P * score::NQ;
  w->above = rank ? reinterpret_cast<int32_t*>(w->gmax) : nullptr;
  w->lo = rank ? w->gmax + Q * nlists : nullptr;
  w->hi = rank ? w->lo + Q : nullptr;
  w->dtarget = rank ? w->hi + Q : nullptr;
  return SEAM_OK;
}

// The tensor maps of the fp16 query and gallery operands and score_topk_kernel's parameters, for either variant.
static int score_kernel_args(seam_handle* h, const ScoreWorkspace& w, int Q, const void* g16, const float* cg, int G,
                             CUtensorMap* tmA, CUtensorMap* tmB, score::Params* sp) {
  int rc;
  if ((rc = encode_map_fp16_rows(h, tmA, w.a16, Q, score::BM)) != SEAM_OK) return rc;
  if ((rc = encode_map_fp16_rows(h, tmB, g16, G, score::BN)) != SEAM_OK) return rc;
  sp->Q = Q;
  sp->G = G;
  sp->P = w.plan.P;
  sp->CAP = w.plan.CAP;
  sp->nseed = w.plan.nseed;
  sp->cg = cg;
  sp->thr_global = w.thr;
  sp->rowcnt = w.rowcnt;
  sp->rowflag = w.rowflag;
  sp->rowbuf = w.rowbuf;
  sp->gmax = w.gmax;
  sp->plan = w.plan.tiles;
  sp->rank_lo = w.lo;
  sp->rank_hi = w.hi;
  sp->rank_above = w.above;
  return SEAM_OK;
}

// rows: the gallery rows of the direct form, of type rt (for fp16 the same pointer as g16).  who names the entry point
// in errors, xwho the sharded entry in the check only a sharded call can fail.
static int score_topk_impl(seam_handle* h, const xchg::Exchange* x, const float* q, int Q, const void* rows,
                           RowType rt, const void* g16, const float* cg, const float* gstat, int G, int index_offset,
                           int k, float* out_score, float* out_margin, int32_t* out_idx, int32_t* stats, void* workspace,
                           size_t workspace_bytes, void* stream_, const char* who, const char* xwho) {
  if (!h->have_scorer) return fail(h, SEAM_ERR_STATE, "%s: scorer weights not loaded", who);
  if (Q < 0 || G < 0) return fail(h, SEAM_ERR_BAD_ARG, "%s: negative size", who);
  if (k < 1 || k > SEAM_MAX_K) return fail(h, SEAM_ERR_UNSUPPORTED, "%s: k=%d outside [1,%d]", who, k, SEAM_MAX_K);
  if (Q == 0 && !x) return SEAM_OK;
  if (!x && (!out_score || !out_margin || !out_idx)) return fail(h, SEAM_ERR_BAD_ARG, "%s: null output", who);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  if (stats) SEAM_CUDA(h, cudaMemsetAsync(stats, 0, 16, stream));
  if (x && (Q == 0 || G == 0))
    return fail(h, SEAM_ERR_UNSUPPORTED, "%s: every rank needs queries and a non-empty gallery shard", xwho);
  const int x_on = x ? 1 : 0;
  xchg::Exchange xe;
  memset(&xe, 0, sizeof(xe));
  if (x) xe = *x;
  if (x) q = x->q_all[x->rank];      // alignment checks below; the kernels pick the step's parity half themselves
  if (G == 0) {
    const size_t n = (size_t)Q * k;
    fill_empty_topk_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(out_score, out_margin, out_idx, n);
    SEAM_LAUNCHED(h, "fill_empty_topk_kernel");
    return SEAM_OK;
  }
  ScoreWorkspace w;
  int rc = carve_score_workspace(h, who, false, q, Q, rows, g16, cg, gstat, G, workspace, workspace_bytes, &w);
  if (rc != SEAM_OK) return rc;

  {
    ProfileScope prof(h, SEAM_KERNEL_PREP_QUERIES, stream);
    exact::prep_queries_kernel<<<(Q + 7) / 8, 256, 0, stream>>>(q, Q, h->fold, w.a16, w.rq, w.anorm, w.thr, w.rowflag,
                                                                w.counters, w.xdone, x_on, xe);
    SEAM_LAUNCHED(h, "prep_queries_kernel");
  }

  CUtensorMap tmA, tmB;
  score::Params sp;
  if ((rc = score_kernel_args(h, w, Q, g16, cg, G, &tmA, &tmB, &sp)) != SEAM_OK) return rc;
  {
    ProfileScope prof(h, SEAM_KERNEL_SCORE, stream);
    score::score_topk_kernel<0><<<w.plan.tiles.nb, score::THREADS, score::SMEM_BYTES, stream>>>(tmA, tmB, sp);
    SEAM_LAUNCHED(h, "score_topk_kernel");
  }

  exact::RescoreParams rp;
  rp.q = q;
  rp.g = rows;
  rp.fold = h->fold;
  rp.rowbuf = w.rowbuf;
  rp.rowcnt = w.rowcnt;
  rp.rowflag = w.rowflag;
  rp.thr_global = w.thr;
  rp.gmax = w.gmax;
  rp.rq = w.rq;
  rp.anorm = w.anorm;
  rp.gstat = gstat;
  rp.Q = Q;
  rp.G = G;
  rp.nlists = w.plan.P * score::NQ;
  rp.CAP = w.plan.CAP;
  rp.k = k;
  rp.index_offset = index_offset;
  rp.out_score = out_score;
  rp.out_margin = out_margin;
  rp.out_idx = out_idx;
  rp.counters = w.counters;
  rp.fallback_rows = w.frows;
  rp.x_on = x_on;
  rp.x = xe;
  rp.plan = w.plan.tiles;
  {
    ProfileScope prof(h, SEAM_KERNEL_RESCORE, stream);
    if (rt == RowType::F16) exact::rescore_kernel<__half><<<(Q + 7) / 8, 256, 0, stream>>>(rp);
    else if (rt == RowType::BF16) exact::rescore_kernel<__nv_bfloat16><<<(Q + 7) / 8, 256, 0, stream>>>(rp);
    else exact::rescore_kernel<float><<<(Q + 7) / 8, 256, 0, stream>>>(rp);
    SEAM_LAUNCHED(h, "rescore_kernel");
  }

  exact::ExactParams ep;
  ep.q = q;
  ep.g = rows;
  ep.fold = h->fold;
  ep.Q = Q;
  ep.G = G;
  ep.k = k;
  ep.index_offset = index_offset;
  ep.count = w.counters;
  ep.rows = w.frows;
  ep.out_score = out_score;
  ep.out_margin = out_margin;
  ep.out_idx = out_idx;
  ep.part_d = w.xpart_d;
  ep.part_i = w.xpart_i;
  ep.done = w.xdone;
  ep.x_on = x_on;
  ep.x = xe;
  {
    ProfileScope prof(h, SEAM_KERNEL_EXACT, stream);
    if (rt == RowType::F16) exact::exact_topk_kernel<__half><<<2 * h->num_sms, 256, 0, stream>>>(ep);
    else if (rt == RowType::BF16) exact::exact_topk_kernel<__nv_bfloat16><<<2 * h->num_sms, 256, 0, stream>>>(ep);
    else exact::exact_topk_kernel<float><<<2 * h->num_sms, 256, 0, stream>>>(ep);
    SEAM_LAUNCHED(h, "exact_topk_kernel");
  }
  if (stats) SEAM_CUDA(h, cudaMemcpyAsync(stats, w.counters, 4, cudaMemcpyDeviceToDevice, stream));
  return SEAM_OK;
}

int seam_score_topk(seam_handle* h, const float* q, int Q, const float* g, const void* g16, const float* cg,
                    const float* gstat, int G, int index_offset, int k, float* out_score, float* out_margin,
                    int32_t* out_idx, int32_t* stats, void* workspace, size_t workspace_bytes, void* stream_) {
  if (!h) return SEAM_ERR_BAD_ARG;
  return score_topk_impl(h, nullptr, q, Q, g, RowType::F32, g16, cg, gstat, G, index_offset, k, out_score, out_margin,
                         out_idx, stats, workspace, workspace_bytes, stream_, "seam_score_topk", "seam_score_topk");
}

int seam_score_topk_g16(seam_handle* h, const float* q, int Q, const void* g16, const float* cg, const float* gstat,
                        int G, int index_offset, int k, float* out_score, float* out_margin, int32_t* out_idx,
                        int32_t* stats, void* workspace, size_t workspace_bytes, void* stream_) {
  if (!h) return SEAM_ERR_BAD_ARG;
  return score_topk_impl(h, nullptr, q, Q, g16, RowType::F16, g16, cg, gstat, G, index_offset, k, out_score, out_margin,
                         out_idx, stats, workspace, workspace_bytes, stream_, "seam_score_topk_g16", "seam_score_topk_g16");
}

int seam_score_topk_gbf16(seam_handle* h, const float* q, int Q, const void* g, const void* g16, const float* cg,
                          const float* gstat, int G, int index_offset, int k, float* out_score, float* out_margin,
                          int32_t* out_idx, int32_t* stats, void* workspace, size_t workspace_bytes, void* stream_) {
  if (!h) return SEAM_ERR_BAD_ARG;
  return score_topk_impl(h, nullptr, q, Q, g, RowType::BF16, g16, cg, gstat, G, index_offset, k, out_score, out_margin,
                         out_idx, stats, workspace, workspace_bytes, stream_, "seam_score_topk_gbf16",
                         "seam_score_topk_gbf16");
}

// tt: the tracks' element type; rows / rt: the gallery rows as in score_topk_impl.  Scorer errors name score_who.
static int search_impl(seam_handle* h, const void* seq, TrackType tt, const uint8_t* mask, const int32_t* lens,
                       int Tmax, int Q, int64_t frame_stride, int64_t track_stride, float* q_out, const void* rows,
                       RowType rt, const void* g16, const float* cg, const float* gstat, int G, int index_offset, int k,
                       float* out_score, float* out_margin, int32_t* out_idx, int32_t* stats, void* workspace,
                       size_t workspace_bytes, void* stream_, const char* who, const char* score_who) {
  if (!h) return SEAM_ERR_BAD_ARG;
  if (!q_out && Q > 0) return fail(h, SEAM_ERR_BAD_ARG, "%s: q_out is null", who);
  int rc = aggregate_impl(h, nullptr, 0, 0, seq, tt, mask, lens, Tmax, Q, frame_stride, track_stride, q_out, nullptr,
                          static_cast<cudaStream_t>(stream_), who);
  if (rc != SEAM_OK) return rc;
  return score_topk_impl(h, nullptr, q_out, Q, rows, rt, g16, cg, gstat, G, index_offset, k, out_score, out_margin,
                         out_idx, stats, workspace, workspace_bytes, stream_, score_who, score_who);
}

int seam_search(seam_handle* h, const float* seq, const uint8_t* mask, const int32_t* lens, int Tmax, int Q,
                int64_t frame_stride, int64_t track_stride, float* q_out, const float* g, const void* g16, const float* cg,
                const float* gstat, int G, int index_offset, int k, float* out_score, float* out_margin, int32_t* out_idx,
                int32_t* stats, void* workspace, size_t workspace_bytes, void* stream_) {
  return search_impl(h, seq, TrackType::F32, mask, lens, Tmax, Q, frame_stride, track_stride, q_out, g, RowType::F32,
                     g16, cg, gstat, G, index_offset, k, out_score, out_margin, out_idx, stats, workspace, workspace_bytes,
                     stream_, "seam_search", "seam_score_topk");
}

int seam_search_f16(seam_handle* h, const void* seq, const uint8_t* mask, const int32_t* lens, int Tmax, int Q,
                    int64_t frame_stride, int64_t track_stride, float* q_out, const float* g, const void* g16,
                    const float* cg, const float* gstat, int G, int index_offset, int k, float* out_score,
                    float* out_margin, int32_t* out_idx, int32_t* stats, void* workspace, size_t workspace_bytes,
                    void* stream_) {
  return search_impl(h, seq, TrackType::F16, mask, lens, Tmax, Q, frame_stride, track_stride, q_out, g, RowType::F32,
                     g16, cg, gstat, G, index_offset, k, out_score, out_margin, out_idx, stats, workspace, workspace_bytes,
                     stream_, "seam_search_f16", "seam_score_topk");
}

int seam_search_bf16(seam_handle* h, const void* seq, const uint8_t* mask, const int32_t* lens, int Tmax, int Q,
                     int64_t frame_stride, int64_t track_stride, float* q_out, const float* g, const void* g16,
                     const float* cg, const float* gstat, int G, int index_offset, int k, float* out_score,
                     float* out_margin, int32_t* out_idx, int32_t* stats, void* workspace, size_t workspace_bytes,
                     void* stream_) {
  return search_impl(h, seq, TrackType::BF16, mask, lens, Tmax, Q, frame_stride, track_stride, q_out, g, RowType::F32,
                     g16, cg, gstat, G, index_offset, k, out_score, out_margin, out_idx, stats, workspace, workspace_bytes,
                     stream_, "seam_search_bf16", "seam_score_topk");
}

int seam_search_g16(seam_handle* h, const float* seq, const uint8_t* mask, const int32_t* lens, int Tmax, int Q,
                    int64_t frame_stride, int64_t track_stride, float* q_out, const void* g16, const float* cg,
                    const float* gstat, int G, int index_offset, int k, float* out_score, float* out_margin,
                    int32_t* out_idx, int32_t* stats, void* workspace, size_t workspace_bytes, void* stream_) {
  return search_impl(h, seq, TrackType::F32, mask, lens, Tmax, Q, frame_stride, track_stride, q_out, g16, RowType::F16,
                     g16, cg, gstat, G, index_offset, k, out_score, out_margin, out_idx, stats, workspace, workspace_bytes,
                     stream_, "seam_search_g16", "seam_search_g16");
}

int seam_search_f16_g16(seam_handle* h, const void* seq, const uint8_t* mask, const int32_t* lens, int Tmax, int Q,
                        int64_t frame_stride, int64_t track_stride, float* q_out, const void* g16, const float* cg,
                        const float* gstat, int G, int index_offset, int k, float* out_score, float* out_margin,
                        int32_t* out_idx, int32_t* stats, void* workspace, size_t workspace_bytes, void* stream_) {
  return search_impl(h, seq, TrackType::F16, mask, lens, Tmax, Q, frame_stride, track_stride, q_out, g16, RowType::F16,
                     g16, cg, gstat, G, index_offset, k, out_score, out_margin, out_idx, stats, workspace, workspace_bytes,
                     stream_, "seam_search_f16_g16", "seam_search_f16_g16");
}

int seam_search_bf16_g16(seam_handle* h, const void* seq, const uint8_t* mask, const int32_t* lens, int Tmax, int Q,
                         int64_t frame_stride, int64_t track_stride, float* q_out, const void* g16, const float* cg,
                         const float* gstat, int G, int index_offset, int k, float* out_score, float* out_margin,
                         int32_t* out_idx, int32_t* stats, void* workspace, size_t workspace_bytes, void* stream_) {
  return search_impl(h, seq, TrackType::BF16, mask, lens, Tmax, Q, frame_stride, track_stride, q_out, g16, RowType::F16,
                     g16, cg, gstat, G, index_offset, k, out_score, out_margin, out_idx, stats, workspace, workspace_bytes,
                     stream_, "seam_search_bf16_g16", "seam_search_bf16_g16");
}

int seam_search_gbf16(seam_handle* h, const float* seq, const uint8_t* mask, const int32_t* lens, int Tmax, int Q,
                      int64_t frame_stride, int64_t track_stride, float* q_out, const void* g, const void* g16,
                      const float* cg, const float* gstat, int G, int index_offset, int k, float* out_score,
                      float* out_margin, int32_t* out_idx, int32_t* stats, void* workspace, size_t workspace_bytes,
                      void* stream_) {
  return search_impl(h, seq, TrackType::F32, mask, lens, Tmax, Q, frame_stride, track_stride, q_out, g, RowType::BF16,
                     g16, cg, gstat, G, index_offset, k, out_score, out_margin, out_idx, stats, workspace, workspace_bytes,
                     stream_, "seam_search_gbf16", "seam_search_gbf16");
}

int seam_search_f16_gbf16(seam_handle* h, const void* seq, const uint8_t* mask, const int32_t* lens, int Tmax, int Q,
                          int64_t frame_stride, int64_t track_stride, float* q_out, const void* g, const void* g16,
                          const float* cg, const float* gstat, int G, int index_offset, int k, float* out_score,
                          float* out_margin, int32_t* out_idx, int32_t* stats, void* workspace, size_t workspace_bytes,
                          void* stream_) {
  return search_impl(h, seq, TrackType::F16, mask, lens, Tmax, Q, frame_stride, track_stride, q_out, g, RowType::BF16,
                     g16, cg, gstat, G, index_offset, k, out_score, out_margin, out_idx, stats, workspace, workspace_bytes,
                     stream_, "seam_search_f16_gbf16", "seam_search_f16_gbf16");
}

int seam_search_bf16_gbf16(seam_handle* h, const void* seq, const uint8_t* mask, const int32_t* lens, int Tmax, int Q,
                           int64_t frame_stride, int64_t track_stride, float* q_out, const void* g, const void* g16,
                           const float* cg, const float* gstat, int G, int index_offset, int k, float* out_score,
                           float* out_margin, int32_t* out_idx, int32_t* stats, void* workspace, size_t workspace_bytes,
                           void* stream_) {
  return search_impl(h, seq, TrackType::BF16, mask, lens, Tmax, Q, frame_stride, track_stride, q_out, g, RowType::BF16,
                     g16, cg, gstat, G, index_offset, k, out_score, out_margin, out_idx, stats, workspace, workspace_bytes,
                     stream_, "seam_search_bf16_gbf16", "seam_search_bf16_gbf16");
}

static int sharded_score_topk_impl(seam_handle* h, const seam_exchange* x, const void* rows, RowType rt,
                                   const void* g16, const float* cg, const float* gstat, int G, int index_offset,
                                   int32_t* stats, void* workspace, size_t workspace_bytes, void* stream_,
                                   const char* who, const char* score_who) {
  if (!h) return SEAM_ERR_BAD_ARG;
  xchg::Exchange e;
  int rc = import_exchange(h, x, &e, who);
  if (rc != SEAM_OK) return rc;
  return score_topk_impl(h, &e, nullptr, x->Q, rows, rt, g16, cg, gstat, G, index_offset, x->k, nullptr, nullptr,
                         nullptr, stats, workspace, workspace_bytes, stream_, score_who, who);
}

int seam_sharded_score_topk(seam_handle* h, const seam_exchange* x, const float* g, const void* g16, const float* cg,
                            const float* gstat, int G, int index_offset, int32_t* stats, void* workspace,
                            size_t workspace_bytes, void* stream_) {
  return sharded_score_topk_impl(h, x, g, RowType::F32, g16, cg, gstat, G, index_offset, stats, workspace, workspace_bytes,
                                 stream_, "seam_sharded_score_topk", "seam_score_topk");
}

int seam_sharded_score_topk_g16(seam_handle* h, const seam_exchange* x, const void* g16, const float* cg,
                                const float* gstat, int G, int index_offset, int32_t* stats, void* workspace,
                                size_t workspace_bytes, void* stream_) {
  return sharded_score_topk_impl(h, x, g16, RowType::F16, g16, cg, gstat, G, index_offset, stats, workspace,
                                 workspace_bytes, stream_, "seam_sharded_score_topk_g16", "seam_sharded_score_topk_g16");
}

int seam_sharded_score_topk_gbf16(seam_handle* h, const seam_exchange* x, const void* g, const void* g16,
                                  const float* cg, const float* gstat, int G, int index_offset, int32_t* stats,
                                  void* workspace, size_t workspace_bytes, void* stream_) {
  return sharded_score_topk_impl(h, x, g, RowType::BF16, g16, cg, gstat, G, index_offset, stats, workspace,
                                 workspace_bytes, stream_, "seam_sharded_score_topk_gbf16",
                                 "seam_sharded_score_topk_gbf16");
}

int seam_sharded_merge(seam_handle* h, const seam_exchange* x, float* out_score, float* out_margin, int32_t* out_idx,
                       void* stream_) {
  if (!h) return SEAM_ERR_BAD_ARG;
  xchg::Exchange e;
  int rc = import_exchange(h, x, &e, "seam_sharded_merge");
  if (rc != SEAM_OK) return rc;
  if (!e.final_score[0] && (!out_score || !out_margin || !out_idx))
    return fail(h, SEAM_ERR_BAD_ARG, "seam_sharded_merge: no final buffers in the exchange and null outputs");
  DeviceGuard guard(h->device);
  const int own = e.q_lo[e.rank + 1] - e.q_lo[e.rank];
  const int grid = own > 0 ? (own + 7) / 8 : 1;
  ProfileScope prof(h, SEAM_KERNEL_MERGE, static_cast<cudaStream_t>(stream_));
  exact::merge_sharded_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream_)>>>(e, out_score, out_margin, out_idx);
  SEAM_LAUNCHED(h, "merge_sharded_kernel");
  return SEAM_OK;
}

int seam_score_dense(seam_handle* h, const float* q, int Q, const float* g, int G, float* x5, void* stream_) {
  if (!h) return SEAM_ERR_BAD_ARG;
  if (!h->have_scorer) return fail(h, SEAM_ERR_STATE, "seam_score_dense: scorer weights not loaded");
  if (Q < 0 || G < 0) return fail(h, SEAM_ERR_BAD_ARG, "seam_score_dense: negative size");
  if (Q == 0 || G == 0) return SEAM_OK;
  if (!q || !g || !x5) return fail(h, SEAM_ERR_BAD_ARG, "seam_score_dense: null pointer");
  if ((reinterpret_cast<uintptr_t>(x5) & 7u)) return fail(h, SEAM_ERR_UNSUPPORTED, "seam_score_dense: x5 alignment");
  DeviceGuard guard(h->device);
  dim3 grid((G + 31) / 32, (Q + 31) / 32);
  if (grid.y > 65535) return fail(h, SEAM_ERR_UNSUPPORTED, "seam_score_dense: Q too large for the dense path");
  exact::dense_logits_kernel<false><<<grid, 256, 0, static_cast<cudaStream_t>(stream_)>>>(q, Q, g, G, h->fold, x5);
  SEAM_LAUNCHED(h, "dense_logits_kernel");
  return SEAM_OK;
}

int seam_score_prob(seam_handle* h, const float* q, int Q, const float* g, int G, float* prob, void* stream_) {
  if (!h) return SEAM_ERR_BAD_ARG;
  if (!h->have_scorer) return fail(h, SEAM_ERR_STATE, "seam_score_prob: scorer weights not loaded");
  if (Q < 0 || G < 0) return fail(h, SEAM_ERR_BAD_ARG, "seam_score_prob: negative size");
  if (Q == 0 || G == 0) return SEAM_OK;
  if (!q || !g || !prob) return fail(h, SEAM_ERR_BAD_ARG, "seam_score_prob: null pointer");
  DeviceGuard guard(h->device);
  dim3 grid((G + 31) / 32, (Q + 31) / 32);
  if (grid.y > 65535) return fail(h, SEAM_ERR_UNSUPPORTED, "seam_score_prob: Q too large for the dense path");
  exact::dense_logits_kernel<true><<<grid, 256, 0, static_cast<cudaStream_t>(stream_)>>>(q, Q, g, G, h->fold, prob);
  SEAM_LAUNCHED(h, "dense_logits_kernel<prob>");
  return SEAM_OK;
}

// rows / rt as in score_topk_impl.  target_avg null: the whole gallery (index_offset 0); else one shard of it,
// counting against the given target values (target[] holds global rows).
static int fused_rank_impl(seam_handle* h, const float* frames, const int32_t* start, int P, const void* rows,
                           RowType rt, int G, int index_offset, const int32_t* target, const float* target_avg,
                           const float* target_max, int32_t* rank_avg, int32_t* rank_max, void* stream_,
                           const char* who) {
  if (!h) return SEAM_ERR_BAD_ARG;
  if (!h->have_scorer) return fail(h, SEAM_ERR_STATE, "%s: scorer weights not loaded", who);
  if (P < 0 || G <= 0) return fail(h, SEAM_ERR_BAD_ARG, "%s: bad size", who);
  if (index_offset < 0) return fail(h, SEAM_ERR_BAD_ARG, "%s: negative index_offset %d", who, index_offset);
  if (P == 0) return SEAM_OK;
  if (!start || !rows || !target || !rank_avg || !rank_max) return fail(h, SEAM_ERR_BAD_ARG, "%s: null pointer", who);
  if ((frames && !aligned16(frames)) || !aligned16(rows)) return fail(h, SEAM_ERR_UNSUPPORTED, "%s: 16-byte alignment", who);
  const int chunks = (G + exact::FD_ROWS - 1) / exact::FD_ROWS;
  if (chunks > 65535) return fail(h, SEAM_ERR_UNSUPPORTED, "%s: G too large", who);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  SEAM_CUDA(h, cudaMemsetAsync(rank_avg, 0, (size_t)P * 4, stream));
  SEAM_CUDA(h, cudaMemsetAsync(rank_max, 0, (size_t)P * 4, stream));
  exact::FusedDistParams fp;
  fp.frames = frames;
  fp.start = start;
  fp.g = rows;
  fp.target = target;
  fp.fold = h->fold;
  fp.P = P;
  fp.G = G;
  fp.rank_avg = rank_avg;
  fp.rank_max = rank_max;
  fp.index_offset = index_offset;
  fp.target_avg = target_avg;
  fp.target_max = target_max;
  const dim3 grid((unsigned)P, (unsigned)chunks);
  if (target_avg) {
    if (rt == RowType::F16) exact::fused_dist_rank_kernel<__half, true><<<grid, 256, 0, stream>>>(fp);
    else if (rt == RowType::BF16) exact::fused_dist_rank_kernel<__nv_bfloat16, true><<<grid, 256, 0, stream>>>(fp);
    else exact::fused_dist_rank_kernel<float, true><<<grid, 256, 0, stream>>>(fp);
  } else {
    if (rt == RowType::F16) exact::fused_dist_rank_kernel<__half, false><<<grid, 256, 0, stream>>>(fp);
    else if (rt == RowType::BF16) exact::fused_dist_rank_kernel<__nv_bfloat16, false><<<grid, 256, 0, stream>>>(fp);
    else exact::fused_dist_rank_kernel<float, false><<<grid, 256, 0, stream>>>(fp);
  }
  SEAM_LAUNCHED(h, "fused_dist_rank_kernel");
  return SEAM_OK;
}

int seam_rank_fused_distances(seam_handle* h, const float* frames, const int32_t* start, int P, const float* g, int G,
                              const int32_t* target, int32_t* rank_avg, int32_t* rank_max, void* stream_) {
  return fused_rank_impl(h, frames, start, P, g, RowType::F32, G, 0, target, nullptr, nullptr, rank_avg, rank_max, stream_,
                         "seam_rank_fused_distances");
}

int seam_rank_fused_distances_g16(seam_handle* h, const float* frames, const int32_t* start, int P, const void* g16,
                                  int G, const int32_t* target, int32_t* rank_avg, int32_t* rank_max, void* stream_) {
  return fused_rank_impl(h, frames, start, P, g16, RowType::F16, G, 0, target, nullptr, nullptr, rank_avg, rank_max,
                         stream_, "seam_rank_fused_distances_g16");
}

int seam_rank_fused_distances_gbf16(seam_handle* h, const float* frames, const int32_t* start, int P, const void* g,
                                    int G, const int32_t* target, int32_t* rank_avg, int32_t* rank_max, void* stream_) {
  return fused_rank_impl(h, frames, start, P, g, RowType::BF16, G, 0, target, nullptr, nullptr, rank_avg, rank_max,
                         stream_, "seam_rank_fused_distances_gbf16");
}

// ------------------------------------------------------------------------------ fusions over a sharded gallery
// rank_p = sum over shards s of #{ j in s : (f_pj, j) ranks before (f_pt, t) } for either fusion f: the owner of row t
// computes the target's fused values (-inf elsewhere, so a MAX all-reduce delivers them to every shard), every shard
// counts against them, and the counts are summed.
static int shard_fused_target_impl(seam_handle* h, const float* frames, const int32_t* start, int P, const void* rows,
                                   RowType rt, int G, int index_offset, const int32_t* target, float* out_avg,
                                   float* out_max, void* stream_, const char* who) {
  if (!h) return SEAM_ERR_BAD_ARG;
  if (!h->have_scorer) return fail(h, SEAM_ERR_STATE, "%s: scorer weights not loaded", who);
  if (P < 0 || G <= 0) return fail(h, SEAM_ERR_BAD_ARG, "%s: bad size", who);
  if (index_offset < 0) return fail(h, SEAM_ERR_BAD_ARG, "%s: negative index_offset %d", who, index_offset);
  if (P == 0) return SEAM_OK;
  if (!start || !rows || !target || !out_avg || !out_max) return fail(h, SEAM_ERR_BAD_ARG, "%s: null pointer", who);
  if ((frames && !aligned16(frames)) || !aligned16(rows)) return fail(h, SEAM_ERR_UNSUPPORTED, "%s: 16-byte alignment", who);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  exact::FusedDistParams fp;
  memset(&fp, 0, sizeof(fp));
  fp.frames = frames;
  fp.start = start;
  fp.g = rows;
  fp.target = target;
  fp.fold = h->fold;
  fp.P = P;
  fp.G = G;
  fp.index_offset = index_offset;
  if (rt == RowType::F16) exact::fused_target_kernel<__half><<<(P + 7) / 8, 256, 0, stream>>>(fp, out_avg, out_max);
  else if (rt == RowType::BF16)
    exact::fused_target_kernel<__nv_bfloat16><<<(P + 7) / 8, 256, 0, stream>>>(fp, out_avg, out_max);
  else exact::fused_target_kernel<float><<<(P + 7) / 8, 256, 0, stream>>>(fp, out_avg, out_max);
  SEAM_LAUNCHED(h, "fused_target_kernel");
  return SEAM_OK;
}

int seam_shard_fused_target(seam_handle* h, const float* frames, const int32_t* start, int P, const float* g, int G,
                            int index_offset, const int32_t* target, float* out_avg, float* out_max, void* stream_) {
  return shard_fused_target_impl(h, frames, start, P, g, RowType::F32, G, index_offset, target, out_avg, out_max, stream_,
                                 "seam_shard_fused_target");
}

int seam_shard_fused_target_g16(seam_handle* h, const float* frames, const int32_t* start, int P, const void* g16,
                                int G, int index_offset, const int32_t* target, float* out_avg, float* out_max,
                                void* stream_) {
  return shard_fused_target_impl(h, frames, start, P, g16, RowType::F16, G, index_offset, target, out_avg, out_max,
                                 stream_, "seam_shard_fused_target_g16");
}

int seam_shard_fused_target_gbf16(seam_handle* h, const float* frames, const int32_t* start, int P, const void* g, int G,
                                  int index_offset, const int32_t* target, float* out_avg, float* out_max,
                                  void* stream_) {
  return shard_fused_target_impl(h, frames, start, P, g, RowType::BF16, G, index_offset, target, out_avg, out_max,
                                 stream_, "seam_shard_fused_target_gbf16");
}

int seam_shard_rank_fused_distances(seam_handle* h, const float* frames, const int32_t* start, int P, const float* g,
                                    int G, int index_offset, const int32_t* target, const float* target_avg,
                                    const float* target_max, int32_t* rank_avg, int32_t* rank_max, void* stream_) {
  if (h && P > 0 && (!target_avg || !target_max))
    return fail(h, SEAM_ERR_BAD_ARG, "seam_shard_rank_fused_distances: null target_avg / target_max");
  return fused_rank_impl(h, frames, start, P, g, RowType::F32, G, index_offset, target, target_avg, target_max, rank_avg,
                         rank_max, stream_, "seam_shard_rank_fused_distances");
}

int seam_shard_rank_fused_distances_g16(seam_handle* h, const float* frames, const int32_t* start, int P,
                                        const void* g16, int G, int index_offset, const int32_t* target,
                                        const float* target_avg, const float* target_max, int32_t* rank_avg,
                                        int32_t* rank_max, void* stream_) {
  if (h && P > 0 && (!target_avg || !target_max))
    return fail(h, SEAM_ERR_BAD_ARG, "seam_shard_rank_fused_distances_g16: null target_avg / target_max");
  return fused_rank_impl(h, frames, start, P, g16, RowType::F16, G, index_offset, target, target_avg, target_max,
                         rank_avg, rank_max, stream_, "seam_shard_rank_fused_distances_g16");
}

int seam_shard_rank_fused_distances_gbf16(seam_handle* h, const float* frames, const int32_t* start, int P,
                                          const void* g, int G, int index_offset, const int32_t* target,
                                          const float* target_avg, const float* target_max, int32_t* rank_avg,
                                          int32_t* rank_max, void* stream_) {
  if (h && P > 0 && (!target_avg || !target_max))
    return fail(h, SEAM_ERR_BAD_ARG, "seam_shard_rank_fused_distances_gbf16: null target_avg / target_max");
  return fused_rank_impl(h, frames, start, P, g, RowType::BF16, G, index_offset, target, target_avg, target_max,
                         rank_avg, rank_max, stream_, "seam_shard_rank_fused_distances_gbf16");
}

int seam_rank_of_target(seam_handle* h, const float* q, int Q, const float* g, int G, const int32_t* target,
                        int32_t* out_rank, float* out_margin, void* stream_) {
  if (!h) return SEAM_ERR_BAD_ARG;
  if (!h->have_scorer) return fail(h, SEAM_ERR_STATE, "seam_rank_of_target: scorer weights not loaded");
  if (Q < 0 || G <= 0) return fail(h, SEAM_ERR_BAD_ARG, "seam_rank_of_target: bad size");
  if (Q == 0) return SEAM_OK;
  if (!q || !g || !target || !out_rank) return fail(h, SEAM_ERR_BAD_ARG, "seam_rank_of_target: null pointer");
  if (!aligned16(q) || !aligned16(g)) return fail(h, SEAM_ERR_UNSUPPORTED, "seam_rank_of_target: 16-byte alignment");
  DeviceGuard guard(h->device);
  exact::rank_of_target_kernel<float, false><<<Q, 256, 0, static_cast<cudaStream_t>(stream_)>>>(
      q, Q, g, G, target, h->fold, nullptr, nullptr, out_rank, out_margin, nullptr, 0);
  SEAM_LAUNCHED(h, "rank_of_target_kernel");
  return SEAM_OK;
}

size_t seam_rank_workspace_bytes(const seam_handle* h, int Q, int G) {
  if (!h || Q <= 0 || G <= 0) return 256;
  return plan_score(h->num_sms, Q, G, true).total;
}

// Tensor-core path: prepare queries -> exact target margins + bands -> score_topk_kernel<VAR_RANK> (counts
// what is certainly above, appends what is inside the band) -> rank_resolve_kernel -> exhaustive kernel for
// the rows that could not be certified.  The workspace is laid out like seam_score_topk's (no sample tiles).
// EXT: one shard of a sharded gallery -- the target margins are given (ext_margin), target[] holds global rows and
// out_rank receives this shard's count of rows ranking before the target.
extern "C++" {   // a template
template <typename Row, bool EXT>
static int rank_launch(seam_handle* h, const ScoreWorkspace& w, const float* q, int Q, const void* rows, const void* g16,
                       const float* cg, const float* gstat, int G, int index_offset, const int32_t* target,
                       const float* ext_margin, int32_t* out_rank, float* out_margin, cudaStream_t stream) {
  const int nlists = w.plan.P * score::NQ;
  const Row* grows = static_cast<const Row*>(rows);
  xchg::Exchange no_x;
  memset(&no_x, 0, sizeof(no_x));
  exact::prep_queries_kernel<<<(Q + 7) / 8, 256, 0, stream>>>(q, Q, h->fold, w.a16, w.rq, w.anorm, w.thr, w.rowflag,
                                                              w.counters, nullptr, 0, no_x);
  SEAM_LAUNCHED(h, "prep_queries_kernel");
  exact::rank_prep_kernel<Row, EXT><<<(Q + 7) / 8, 256, 0, stream>>>(q, Q, grows, target, h->fold, w.rq, w.anorm, gstat,
                                                                     w.lo, w.hi, w.dtarget, w.above, nlists, ext_margin);
  SEAM_LAUNCHED(h, "rank_prep_kernel");

  CUtensorMap tmA, tmB;
  score::Params sp;
  int rc;
  if ((rc = score_kernel_args(h, w, Q, g16, cg, G, &tmA, &tmB, &sp)) != SEAM_OK) return rc;
  score::score_topk_kernel<score::VAR_RANK><<<w.plan.tiles.nb, score::THREADS, score::SMEM_BYTES, stream>>>(tmA, tmB, sp);
  SEAM_LAUNCHED(h, "score_topk_kernel<rank>");

  exact::RankResolveParams rp;
  rp.q = q;
  rp.g = rows;
  rp.fold = h->fold;
  rp.rowbuf = w.rowbuf;
  rp.rowcnt = w.rowcnt;
  rp.rowflag = w.rowflag;
  rp.above = w.above;
  rp.lo = w.lo;
  rp.hi = w.hi;
  rp.dtarget = w.dtarget;
  rp.rq = w.rq;
  rp.gstat = gstat;
  rp.target = target;
  rp.Q = Q;
  rp.G = G;
  rp.nlists = nlists;
  rp.CAP = w.plan.CAP;
  rp.out_rank = out_rank;
  rp.out_margin = out_margin;
  rp.counters = w.counters;
  rp.fallback_rows = w.frows;
  rp.plan = w.plan.tiles;
  rp.index_offset = index_offset;
  exact::rank_resolve_kernel<Row, EXT><<<(Q + 7) / 8, 256, 0, stream>>>(rp);
  SEAM_LAUNCHED(h, "rank_resolve_kernel");
  exact::rank_of_target_kernel<Row, EXT><<<2 * h->num_sms, 256, 0, stream>>>(q, Q, grows, G, target, h->fold, w.counters,
                                                                             w.frows, out_rank, out_margin, ext_margin,
                                                                             index_offset);
  SEAM_LAUNCHED(h, "rank_of_target_kernel");
  return SEAM_OK;
}
}  // extern "C++"

// rows / rt as in score_topk_impl.  ext_margin null: the whole gallery (index_offset 0, out_margin optional);
// else one shard of it, counting against the given target margins (out_margin null).
static int rank_prepared_impl(seam_handle* h, const float* q, int Q, const void* rows, RowType rt, const void* g16,
                              const float* cg, const float* gstat, int G, int index_offset, const int32_t* target,
                              const float* ext_margin, int32_t* out_rank, float* out_margin, int32_t* stats,
                              void* workspace, size_t workspace_bytes, void* stream_, const char* who) {
  if (!h) return SEAM_ERR_BAD_ARG;
  if (!h->have_scorer) return fail(h, SEAM_ERR_STATE, "%s: scorer weights not loaded", who);
  if (Q < 0 || G <= 0) return fail(h, SEAM_ERR_BAD_ARG, "%s: bad size", who);
  if (index_offset < 0) return fail(h, SEAM_ERR_BAD_ARG, "%s: negative index_offset %d", who, index_offset);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  if (stats) SEAM_CUDA(h, cudaMemsetAsync(stats, 0, 16, stream));
  if (Q == 0) return SEAM_OK;
  if (!target || !out_rank) return fail(h, SEAM_ERR_BAD_ARG, "%s: null pointer", who);
  ScoreWorkspace w;
  int rc = carve_score_workspace(h, who, true, q, Q, rows, g16, cg, gstat, G, workspace, workspace_bytes, &w);
  if (rc != SEAM_OK) return rc;
  if (ext_margin) {
    if (rt == RowType::F16)
      rc = rank_launch<__half, true>(h, w, q, Q, rows, g16, cg, gstat, G, index_offset, target, ext_margin, out_rank,
                                     nullptr, stream);
    else if (rt == RowType::BF16)
      rc = rank_launch<__nv_bfloat16, true>(h, w, q, Q, rows, g16, cg, gstat, G, index_offset, target, ext_margin,
                                            out_rank, nullptr, stream);
    else
      rc = rank_launch<float, true>(h, w, q, Q, rows, g16, cg, gstat, G, index_offset, target, ext_margin, out_rank,
                                    nullptr, stream);
  } else {
    if (rt == RowType::F16)
      rc = rank_launch<__half, false>(h, w, q, Q, rows, g16, cg, gstat, G, 0, target, nullptr, out_rank, out_margin,
                                      stream);
    else if (rt == RowType::BF16)
      rc = rank_launch<__nv_bfloat16, false>(h, w, q, Q, rows, g16, cg, gstat, G, 0, target, nullptr, out_rank,
                                             out_margin, stream);
    else
      rc = rank_launch<float, false>(h, w, q, Q, rows, g16, cg, gstat, G, 0, target, nullptr, out_rank, out_margin,
                                     stream);
  }
  if (rc != SEAM_OK) return rc;
  if (stats) SEAM_CUDA(h, cudaMemcpyAsync(stats, w.counters, 4, cudaMemcpyDeviceToDevice, stream));
  return SEAM_OK;
}

int seam_rank_of_target_prepared(seam_handle* h, const float* q, int Q, const float* g, const void* g16,
                                 const float* cg, const float* gstat, int G, const int32_t* target, int32_t* out_rank,
                                 float* out_margin, int32_t* stats, void* workspace, size_t workspace_bytes,
                                 void* stream_) {
  return rank_prepared_impl(h, q, Q, g, RowType::F32, g16, cg, gstat, G, 0, target, nullptr, out_rank, out_margin, stats,
                            workspace, workspace_bytes, stream_, "seam_rank_of_target_prepared");
}

int seam_rank_of_target_prepared_g16(seam_handle* h, const float* q, int Q, const void* g16, const float* cg,
                                     const float* gstat, int G, const int32_t* target, int32_t* out_rank,
                                     float* out_margin, int32_t* stats, void* workspace, size_t workspace_bytes,
                                     void* stream_) {
  return rank_prepared_impl(h, q, Q, g16, RowType::F16, g16, cg, gstat, G, 0, target, nullptr, out_rank, out_margin,
                            stats, workspace, workspace_bytes, stream_, "seam_rank_of_target_prepared_g16");
}

int seam_rank_of_target_prepared_gbf16(seam_handle* h, const float* q, int Q, const void* g, const void* g16,
                                       const float* cg, const float* gstat, int G, const int32_t* target,
                                       int32_t* out_rank, float* out_margin, int32_t* stats, void* workspace,
                                       size_t workspace_bytes, void* stream_) {
  return rank_prepared_impl(h, q, Q, g, RowType::BF16, g16, cg, gstat, G, 0, target, nullptr, out_rank, out_margin,
                            stats, workspace, workspace_bytes, stream_, "seam_rank_of_target_prepared_gbf16");
}

// ------------------------------------------------------------------------------ rank over a sharded gallery
// rank_i = sum over shards s of #{ j in s : (d_ij, j) ranks before (d_it, t) }: the owner of row t computes the
// target's margin (-inf elsewhere, so a MAX all-reduce delivers it to every shard), every shard counts against it, and
// the counts are summed.
static int shard_target_margin_impl(seam_handle* h, const float* q, int Q, const void* rows, RowType rt, int G,
                                    int index_offset, const int32_t* target, float* out_margin, void* stream_,
                                    const char* who) {
  if (!h) return SEAM_ERR_BAD_ARG;
  if (!h->have_scorer) return fail(h, SEAM_ERR_STATE, "%s: scorer weights not loaded", who);
  if (Q < 0 || G <= 0) return fail(h, SEAM_ERR_BAD_ARG, "%s: bad size", who);
  if (index_offset < 0) return fail(h, SEAM_ERR_BAD_ARG, "%s: negative index_offset %d", who, index_offset);
  if (Q == 0) return SEAM_OK;
  if (!q || !rows || !target || !out_margin) return fail(h, SEAM_ERR_BAD_ARG, "%s: null pointer", who);
  if (!aligned16(q) || !aligned16(rows)) return fail(h, SEAM_ERR_UNSUPPORTED, "%s: q/g need 16-byte alignment", who);
  DeviceGuard guard(h->device);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (rt == RowType::F16)
    exact::target_margin_kernel<__half><<<(Q + 7) / 8, 256, 0, stream>>>(q, Q, static_cast<const __half*>(rows), G,
                                                                         index_offset, target, h->fold, out_margin);
  else if (rt == RowType::BF16)
    exact::target_margin_kernel<__nv_bfloat16><<<(Q + 7) / 8, 256, 0, stream>>>(
        q, Q, static_cast<const __nv_bfloat16*>(rows), G, index_offset, target, h->fold, out_margin);
  else
    exact::target_margin_kernel<float><<<(Q + 7) / 8, 256, 0, stream>>>(q, Q, static_cast<const float*>(rows), G,
                                                                        index_offset, target, h->fold, out_margin);
  SEAM_LAUNCHED(h, "target_margin_kernel");
  return SEAM_OK;
}

int seam_shard_target_margin(seam_handle* h, const float* q, int Q, const float* g, int G, int index_offset,
                             const int32_t* target, float* out_margin, void* stream_) {
  return shard_target_margin_impl(h, q, Q, g, RowType::F32, G, index_offset, target, out_margin, stream_,
                                  "seam_shard_target_margin");
}

int seam_shard_target_margin_g16(seam_handle* h, const float* q, int Q, const void* g16, int G, int index_offset,
                                 const int32_t* target, float* out_margin, void* stream_) {
  return shard_target_margin_impl(h, q, Q, g16, RowType::F16, G, index_offset, target, out_margin, stream_,
                                  "seam_shard_target_margin_g16");
}

int seam_shard_target_margin_gbf16(seam_handle* h, const float* q, int Q, const void* g, int G, int index_offset,
                                   const int32_t* target, float* out_margin, void* stream_) {
  return shard_target_margin_impl(h, q, Q, g, RowType::BF16, G, index_offset, target, out_margin, stream_,
                                  "seam_shard_target_margin_gbf16");
}

int seam_shard_rank_count_prepared(seam_handle* h, const float* q, int Q, const float* g, const void* g16,
                                   const float* cg, const float* gstat, int G, int index_offset, const int32_t* target,
                                   const float* target_margin, int32_t* out_count, int32_t* stats, void* workspace,
                                   size_t workspace_bytes, void* stream_) {
  if (h && Q > 0 && !target_margin)
    return fail(h, SEAM_ERR_BAD_ARG, "seam_shard_rank_count_prepared: null target_margin");
  return rank_prepared_impl(h, q, Q, g, RowType::F32, g16, cg, gstat, G, index_offset, target, target_margin, out_count,
                            nullptr, stats, workspace, workspace_bytes, stream_, "seam_shard_rank_count_prepared");
}

int seam_shard_rank_count_prepared_g16(seam_handle* h, const float* q, int Q, const void* g16, const float* cg,
                                       const float* gstat, int G, int index_offset, const int32_t* target,
                                       const float* target_margin, int32_t* out_count, int32_t* stats,
                                       void* workspace, size_t workspace_bytes, void* stream_) {
  if (h && Q > 0 && !target_margin)
    return fail(h, SEAM_ERR_BAD_ARG, "seam_shard_rank_count_prepared_g16: null target_margin");
  return rank_prepared_impl(h, q, Q, g16, RowType::F16, g16, cg, gstat, G, index_offset, target, target_margin,
                            out_count, nullptr, stats, workspace, workspace_bytes, stream_,
                            "seam_shard_rank_count_prepared_g16");
}

int seam_shard_rank_count_prepared_gbf16(seam_handle* h, const float* q, int Q, const void* g, const void* g16,
                                         const float* cg, const float* gstat, int G, int index_offset,
                                         const int32_t* target, const float* target_margin, int32_t* out_count,
                                         int32_t* stats, void* workspace, size_t workspace_bytes, void* stream_) {
  if (h && Q > 0 && !target_margin)
    return fail(h, SEAM_ERR_BAD_ARG, "seam_shard_rank_count_prepared_gbf16: null target_margin");
  return rank_prepared_impl(h, q, Q, g, RowType::BF16, g16, cg, gstat, G, index_offset, target, target_margin,
                            out_count, nullptr, stats, workspace, workspace_bytes, stream_,
                            "seam_shard_rank_count_prepared_gbf16");
}

// ------------------------------------------------------------------------------ backward (f4)
int seam_aggregate_backward(seam_handle* h, const seam_weights* w, const float* seq, const uint8_t* mask,
                            const int32_t* lens, int Tmax, int Q, int64_t frame_stride, int64_t track_stride,
                            const float* dout, float* dseq, const seam_weight_grads* grads, void* stream_) {
  if (!h) return SEAM_ERR_BAD_ARG;
  if (!w || !grads) return fail(h, SEAM_ERR_BAD_ARG, "seam_aggregate_backward: weights / grads struct is null");
  if (Q < 0 || Tmax < 0) return fail(h, SEAM_ERR_BAD_ARG, "seam_aggregate_backward: negative size");
  if (Q == 0 || Tmax == 0) return SEAM_OK;
  if (Tmax > SEAM_MAX_T)
    return fail(h, SEAM_ERR_UNSUPPORTED, "seam_aggregate_backward: Tmax=%d exceeds %d", Tmax, SEAM_MAX_T);
  if (!seq || !dout || !dseq) return fail(h, SEAM_ERR_BAD_ARG, "seam_aggregate_backward: null pointer");
  const float* const* wp = reinterpret_cast<const float* const*>(w);
  float* const* gp = reinterpret_cast<float* const*>(grads);
  for (int i = 0; i < 11; ++i)
    if (!wp[i] || !gp[i]) return fail(h, SEAM_ERR_BAD_ARG, "seam_aggregate_backward: null weight / gradient pointer %d", i);
  DeviceGuard guard(h->device);
  bwd::AggBwdParams p;
  p.seq = seq;
  p.mask = mask;
  p.lens = lens;
  p.Tmax = Tmax;
  p.Q = Q;
  p.frame_stride = frame_stride;
  p.track_stride = track_stride;
  p.dout = dout;
  p.dseq = dseq;
  p.w = {w->theta_w, w->theta_b, w->phi_w, w->phi_b, w->g_w, w->g_b, w->W_w, w->W_b, w->concat_w, w->att_w, w->att_b};
  p.g = {grads->theta_w, grads->theta_b, grads->phi_w, grads->phi_b, grads->g_w, grads->g_b,
         grads->W_w,     grads->W_b,     grads->concat_w, grads->att_w, grads->att_b};
  // persistent CTAs: each folds the weights once, so no more of them than can be resident at once
  const size_t smem = bwd::agg_bwd_smem_bytes(Tmax);
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, bwd::agg_backward_folded_kernel, 256, smem) != cudaSuccess ||
      per_sm < 1)
    return fail(h, SEAM_ERR_CUDA, "seam_aggregate_backward: occupancy query failed: %s", cudaGetErrorString(cudaGetLastError()));
  const int grid = Q < per_sm * h->num_sms ? Q : per_sm * h->num_sms;
  bwd::agg_backward_folded_kernel<<<grid, 256, smem, static_cast<cudaStream_t>(stream_)>>>(p);
  SEAM_LAUNCHED(h, "agg_backward_folded_kernel");
  return SEAM_OK;
}

int seam_score_dense_backward(seam_handle* h, const float* last_w, const float* q, int Q, const float* g, int G,
                              const float* dx5, float* dq, float* dg, float* dlast_w, float* dlast_b, void* stream_) {
  if (!h) return SEAM_ERR_BAD_ARG;
  if (Q < 0 || G < 0) return fail(h, SEAM_ERR_BAD_ARG, "seam_score_dense_backward: negative size");
  if (Q == 0 || G == 0) return SEAM_OK;
  if (!last_w || !q || !g || !dx5 || !dq || !dg || !dlast_w || !dlast_b)
    return fail(h, SEAM_ERR_BAD_ARG, "seam_score_dense_backward: null pointer");
  if ((reinterpret_cast<uintptr_t>(dx5) & 7u)) return fail(h, SEAM_ERR_UNSUPPORTED, "seam_score_dense_backward: dx5 alignment");
  DeviceGuard guard(h->device);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  bwd::scorer_backward_q_kernel<<<Q, 256, 0, stream>>>(q, Q, g, G, last_w, dx5, dq, dlast_w, dlast_b);
  SEAM_LAUNCHED(h, "scorer_backward_q_kernel");
  bwd::scorer_backward_g_kernel<<<G, 256, 0, stream>>>(q, Q, g, G, last_w, dx5, dg);
  SEAM_LAUNCHED(h, "scorer_backward_g_kernel");
  return SEAM_OK;
}

// ------------------------------------------------------------------------------ conv tower (f3)
namespace {
constexpr int TW_GUARD = 192;                                    // rows a shifted A box may reach past a layer's last position
constexpr size_t TW_OFF_B[4] = {0, 256, 512, 768};               // biases inside tw_misc (floats)
constexpr size_t TW_OFF_WT = 1792, TW_OFF_LB = TW_OFF_WT + 1024 * 256, TW_OFF_SC = TW_OFF_LB + 256,
                 TW_OFF_SH = TW_OFF_SC + 256, TW_MISC_TOTAL = TW_OFF_SH + 256;
const int TW_HW[5] = {14, 12, 10, 8, 6};
struct TowerPlan {
  size_t off[5], total;
};
TowerPlan plan_tower(int K) {
  TowerPlan t;
  size_t o = 0;
  for (int l = 0; l < 5; ++l) {
    t.off[l] = o;
    const size_t rows = (size_t)K * TW_HW[l] * TW_HW[l] + (l < 4 ? TW_GUARD : 0);
    o += align_up(rows * (l < 4 ? 256 : 1024) * 2, 1024);
  }
  t.total = o;
  return t;
}
int encode_map_fp16_2d(seam_handle* h, CUtensorMap* map, const void* base, uint64_t inner, uint64_t rows, uint32_t box_rows) {
  const cuuint64_t dims[2] = {inner, rows};
  const cuuint64_t strides[1] = {inner * 2};
  const cuuint32_t box[2] = {(cuuint32_t)tower::BK, box_rows};
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = h->encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(h, SEAM_ERR_CUDA, "cuTensorMapEncodeTiled (tower) failed with CUresult %d", (int)r);
  return SEAM_OK;
}
}  // namespace

int seam_tower_load_weights(seam_handle* h, const float* const* conv_w, const float* const* conv_b, const float* lin_w,
                            const float* lin_b, const float* bn_gamma, const float* bn_beta, const float* bn_mean,
                            const float* bn_var, float bn_eps, void* stream_) {
  if (!h) return SEAM_ERR_BAD_ARG;
  if (!conv_w || !conv_b || !lin_w || !lin_b || !bn_gamma || !bn_beta || !bn_mean || !bn_var)
    return fail(h, SEAM_ERR_BAD_ARG, "seam_tower_load_weights: null pointer");
  for (int l = 0; l < 4; ++l)
    if (!conv_w[l] || !conv_b[l]) return fail(h, SEAM_ERR_BAD_ARG, "seam_tower_load_weights: null conv parameter %d", l);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  for (int l = 0; l < 4; ++l) {
    const int cout = l < 3 ? 256 : 1024;
    if (!h->tw_conv[l]) SEAM_CUDA(h, cudaMalloc(&h->tw_conv[l], (size_t)cout * 2304 * 2));
  }
  if (!h->tw_misc) SEAM_CUDA(h, cudaMalloc(&h->tw_misc, TW_MISC_TOTAL * 4));
  for (int l = 0; l < 4; ++l) {
    const int cout = l < 3 ? 256 : 1024;
    tower::conv_weight_rows_kernel<<<cout, 256, 0, stream>>>(conv_w[l], h->tw_conv[l], cout);
    SEAM_LAUNCHED(h, "conv_weight_rows_kernel");
    SEAM_CUDA(h, cudaMemcpyAsync(h->tw_misc + TW_OFF_B[l], conv_b[l], (size_t)cout * 4, cudaMemcpyDeviceToDevice, stream));
  }
  SEAM_CUDA(h, cudaMemcpyAsync(h->tw_misc + TW_OFF_LB, lin_b, 256 * 4, cudaMemcpyDeviceToDevice, stream));
  tower::tower_fold_kernel<<<256, 256, 0, stream>>>(lin_w, bn_gamma, bn_beta, bn_mean, bn_var, bn_eps, h->tw_misc + TW_OFF_WT,
                                                    h->tw_misc + TW_OFF_SC, h->tw_misc + TW_OFF_SH);
  SEAM_LAUNCHED(h, "tower_fold_kernel");
  h->have_tower = true;
  return SEAM_OK;
}

size_t seam_tower_workspace_bytes(int K) { return K > 0 ? plan_tower(K).total : 1024; }

int seam_tower_forward(seam_handle* h, const float* x, int K, float* out, const int64_t* dst_row, void* workspace,
                       size_t workspace_bytes, void* stream_) {
  if (!h) return SEAM_ERR_BAD_ARG;
  if (!h->have_tower) return fail(h, SEAM_ERR_STATE, "seam_tower_forward: tower weights not loaded");
  if (K < 0) return fail(h, SEAM_ERR_BAD_ARG, "seam_tower_forward: negative size");
  if (K == 0) return SEAM_OK;
  if ((long long)K * 196 > 0x7fffff00ll) return fail(h, SEAM_ERR_UNSUPPORTED, "seam_tower_forward: K too large");
  if (!x || !out || !workspace) return fail(h, SEAM_ERR_BAD_ARG, "seam_tower_forward: null pointer");
  if ((reinterpret_cast<uintptr_t>(workspace) & 1023u)) return fail(h, SEAM_ERR_UNSUPPORTED, "seam_tower_forward: workspace must be 1 KB aligned");
  const TowerPlan tp = plan_tower(K);
  if (workspace_bytes < tp.total) return fail(h, SEAM_ERR_STATE, "seam_tower_forward: workspace too small (%zu < %zu)", workspace_bytes, tp.total);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DeviceGuard guard(h->device);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  ProfileScope prof(h, SEAM_KERNEL_TOWER, stream);
  tower::nchw_to_rows_kernel<<<dim3((unsigned)K, 8), 256, 0, stream>>>(x, reinterpret_cast<__half*>(ws + tp.off[0]), K);
  SEAM_LAUNCHED(h, "nchw_to_rows_kernel");
  for (int l = 0; l < 4; ++l) {
    const int H = TW_HW[l], cout = l < 3 ? 256 : 1024;
    const long long rows_in = (long long)K * H * H;
    CUtensorMap tmA, tmB;
    int rc;
    if ((rc = encode_map_fp16_2d(h, &tmA, ws + tp.off[l], 256, (uint64_t)rows_in + TW_GUARD, tower::BM)) != SEAM_OK) return rc;
    if ((rc = encode_map_fp16_2d(h, &tmB, h->tw_conv[l], 2304, (uint64_t)cout, tower::BN)) != SEAM_OK) return rc;
    tower::ConvParams cp;
    cp.H = H;
    cp.W = H;
    cp.K = K;
    cp.Cout = cout;
    cp.rows_in = rows_in;
    cp.m_tiles = (int)((rows_in + tower::BM - 1) / tower::BM);
    cp.n_tiles = cout / tower::BN;
    cp.bias = h->tw_misc + TW_OFF_B[l];
    cp.out = reinterpret_cast<__half*>(ws + tp.off[l + 1]);
    const long long total = (long long)cp.m_tiles * cp.n_tiles;
    const int grid = total < h->num_sms ? (int)total : h->num_sms;
    tower::conv3x3_kernel<<<grid, tower::THREADS, tower::SMEM_BYTES, stream>>>(tmA, tmB, cp);
    SEAM_LAUNCHED(h, "conv3x3_kernel");
  }
  tower::PoolLinearParams pp;
  pp.a4 = reinterpret_cast<const __half*>(ws + tp.off[4]);
  pp.wt = h->tw_misc + TW_OFF_WT;
  pp.lin_b = h->tw_misc + TW_OFF_LB;
  pp.bn_scale = h->tw_misc + TW_OFF_SC;
  pp.bn_shift = h->tw_misc + TW_OFF_SH;
  pp.dst_row = reinterpret_cast<const long long*>(dst_row);
  pp.out = out;
  pp.K = K;
  tower::pool_linear_bn_kernel<<<(K + tower::PL_ROIS - 1) / tower::PL_ROIS, 256, 0, stream>>>(pp);
  SEAM_LAUNCHED(h, "pool_linear_bn_kernel");
  return SEAM_OK;
}

// es: bytes per element (4: fp32, 2: fp16 or bf16); a frame row of one track is 256 * es bytes
static int upload_tracks_impl(seam_handle* h, const void* seq_host, size_t es, int Tmax, int Q, int lo, int hi,
                              void* seq_dev, void* stream_, const char* who) {
  if (!h) return SEAM_ERR_BAD_ARG;
  if (Tmax < 0 || Q < 0 || lo < 0 || hi < lo || hi > Q) return fail(h, SEAM_ERR_BAD_ARG, "%s: bad range", who);
  if (Tmax == 0 || hi == lo) return SEAM_OK;
  if (!seq_host || !seq_dev) return fail(h, SEAM_ERR_BAD_ARG, "%s: null pointer", who);
  DeviceGuard guard(h->device);
  const size_t n = (size_t)(hi - lo), row = 256 * es;
  SEAM_CUDA(h, cudaMemcpy2DAsync(static_cast<uint8_t*>(seq_dev) + n * row, n * row,
                                 static_cast<const uint8_t*>(seq_host) + ((size_t)Q + (size_t)lo) * row, (size_t)Q * row,
                                 n * row, (size_t)Tmax, cudaMemcpyHostToDevice, static_cast<cudaStream_t>(stream_)));
  return SEAM_OK;
}

int seam_upload_tracks(seam_handle* h, const float* seq_host, int Tmax, int Q, int lo, int hi, float* seq_dev,
                       void* stream_) {
  return upload_tracks_impl(h, seq_host, 4, Tmax, Q, lo, hi, seq_dev, stream_, "seam_upload_tracks");
}

int seam_upload_tracks_f16(seam_handle* h, const void* seq_host, int Tmax, int Q, int lo, int hi, void* seq_dev,
                           void* stream_) {
  return upload_tracks_impl(h, seq_host, 2, Tmax, Q, lo, hi, seq_dev, stream_, "seam_upload_tracks_f16");
}

int seam_merge_topk(seam_handle* h, const float* scores, const float* margins, const int32_t* idx, int N, int Q,
                    int k, float* out_score, float* out_margin, int32_t* out_idx, void* stream_) {
  if (!h) return SEAM_ERR_BAD_ARG;
  if (N < 1 || Q < 0) return fail(h, SEAM_ERR_BAD_ARG, "seam_merge_topk: bad size");
  if (k < 1 || k > SEAM_MAX_K) return fail(h, SEAM_ERR_UNSUPPORTED, "seam_merge_topk: k=%d outside [1,%d]", k, SEAM_MAX_K);
  if (Q == 0) return SEAM_OK;
  if (!margins || !idx || !out_score || !out_margin || !out_idx)    // scores may be null: recomputed from the margins
    return fail(h, SEAM_ERR_BAD_ARG, "seam_merge_topk: null pointer");
  DeviceGuard guard(h->device);
  ProfileScope prof(h, SEAM_KERNEL_MERGE, static_cast<cudaStream_t>(stream_));
  exact::merge_topk_kernel<<<(Q + 7) / 8, 256, 0, static_cast<cudaStream_t>(stream_)>>>(
      scores, margins, idx, N, Q, k, out_score, out_margin, out_idx);
  SEAM_LAUNCHED(h, "merge_topk_kernel");
  return SEAM_OK;
}

}  // extern "C"
