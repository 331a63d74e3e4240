// Shared device/host helpers for librr_sm100 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <mutex>
#include <stdint.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>
#include <utility>

#include "rr_sm100.h"

namespace rr {

// ---- error plumbing (no exceptions cross the C ABI) ----------------------------------
extern thread_local char g_err[512];
extern std::atomic<int64_t> g_launches;   // process-wide: autograd runs backward on its own thread

inline int fail(int code, const char* fmt, ...) __attribute__((format(printf, 2, 3)));
inline int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define RR_CUDA(expr)                                                                         \
  do {                                                                                        \
    cudaError_t _e = (expr);                                                                  \
    if (_e != cudaSuccess) return rr::fail(RR_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(_e)); \
  } while (0)

#define RR_LAUNCH_CHECK(name)                                                                 \
  do {                                                                                        \
    ++rr::g_launches;                                                                         \
    cudaError_t _e = cudaGetLastError();                                                      \
    if (_e != cudaSuccess) return rr::fail(RR_ERR_CUDA, "launch %s: %s", name, cudaGetErrorString(_e)); \
  } while (0)

// ---- optional per-kernel-class timing with CUDA events on the launching stream (bench.py) ----
enum KernelClass { KC_GEMM_FWD = 0, KC_GEMM_DGRAD, KC_GEMM_WGRAD, KC_BOND_FWD, KC_BOND_BWD, KC_NBR_FWD, KC_NBR_BWD, KC_READOUT,
                   KC_ELEMENTWISE, KC_LOSS, KC_MISC, KC_COUNT };
struct ProfState {
  bool enabled = false;
  struct Rec { int cls; cudaEvent_t a, b; };
  Rec* recs = nullptr;
  int n = 0, cap = 0;
};
extern ProfState g_prof;  // process-wide, guarded by g_prof_mutex
extern std::mutex g_prof_mutex;
void prof_push(int cls, cudaEvent_t a, cudaEvent_t b);
struct ProfScope {
  cudaEvent_t a = nullptr, b = nullptr;
  cudaStream_t s;
  int cls;
  ProfScope(int cls_, cudaStream_t s_) : s(s_), cls(cls_) {
    if (g_prof.enabled) {
      cudaEventCreate(&a);
      cudaEventCreate(&b);
      cudaEventRecord(a, s);
    }
  }
  ~ProfScope() {
    if (a) {
      cudaEventRecord(b, s);
      prof_push(cls, a, b);
    }
  }
};

// Precision switches of the dense layers (rr_set_gemm_mode / _backward_bf16 / _forward_bf16), read only by rr_linear.cu, whose header
// comment gives the policy they select
extern std::atomic<int> g_gemm_mode;
extern std::atomic<int> g_fwd_bf16;
extern std::atomic<int> g_bwd_bf16;

// Deterministic mode (rr_set_deterministic): every sum the backward pass and the losses would form with atomics is instead written as
// partials to scratch with plain stores and summed in a fixed order.  Process-wide.
extern std::atomic<int> g_deterministic;
inline bool deterministic() { return g_deterministic.load() != 0; }

// Scratch of a deterministic launch: the caller's (the model's workspace) when given, else transient stream-ordered memory that is freed on
// the same stream once the launches that use it are enqueued, so the library still holds nothing between calls.
struct DetScratch {
  void* p = nullptr;
  cudaStream_t s = nullptr;
  bool owned = false;
  DetScratch() = default;
  DetScratch(const DetScratch&) = delete;
  DetScratch& operator=(const DetScratch&) = delete;
  ~DetScratch() {
    if (owned) cudaFreeAsync(p, s);
  }
};

// Switches from the environment (RR_MP_V1: the first-generation gather kernels instead of the row pipeline): read ONCE, when the library is
// first used, not on every launch.  rr_reload_switches() reads them again (tests and the micro-benchmarks flip them inside one process).
struct Switches {
  int mp_v1 = 0;
};
const Switches& switches();
void reload_switches();

#define RR_REQUIRE(cond, ...)                                  \
  do {                                                         \
    if (!(cond)) return rr::fail(RR_ERR_INVALID, __VA_ARGS__); \
  } while (0)

#define RR_TRY(expr)          \
  do {                        \
    int _s = (expr);          \
    if (_s != RR_OK) return _s; \
  } while (0)

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
inline int check_mat(const char* what, const void* p, int ld) {
  RR_REQUIRE(p != nullptr, "%s is NULL", what);
  RR_REQUIRE(aligned16(p) && (ld & 3) == 0, "%s must be 16-byte aligned with a row stride multiple of 4 (ld %d)", what, ld);
  return RR_OK;
}
constexpr int kMaxDevices = 64;
inline int current_device() {
  int dev = 0;
  cudaGetDevice(&dev);
  return (dev >= 0 && dev < kMaxDevices) ? dev : 0;
}
// cached per device: one process may drive several GPUs through the `gpu` argument of the Python API
inline int num_sms() {
  static int n[kMaxDevices] = {};
  const int dev = current_device();
  if (n[dev] == 0) {
    cudaDeviceGetAttribute(&n[dev], cudaDevAttrMultiProcessorCount, dev);
    if (n[dev] <= 0) n[dev] = 148;
  }
  return n[dev];
}
// cudaFuncSetAttribute is per device (per context): remember where a kernel's dynamic shared-memory limit has been raised
struct PerDeviceOnce {
  bool done[kMaxDevices] = {};
  bool need() const { return !done[current_device()]; }
  void mark() { done[current_device()] = true; }
};

// ---- programmatic dependent launch -------------------------------------------------------
// The big kernels are persistent, one CTA per SM, with a prologue of a few microseconds (barrier init, TMEM allocation, descriptor prefetch).
// Launched with cudaLaunchAttributeProgrammaticStreamSerialization, the CTAs of kernel N+1 start on every SM that kernel N has left and run
// their prologue while N's tail still executes; pdl_wait() (griddepcontrol.wait) then holds every thread until kernel N has completed and
// its writes are visible, BEFORE the first global access of N+1 (reads and writes alike).
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// ---- float4 helpers ---------------------------------------------------------------------
__device__ __forceinline__ float4 f4_zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ float4 f4_add(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
__device__ __forceinline__ float4 f4_sub(float4 a, float4 b) { return make_float4(a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w); }
__device__ __forceinline__ float4 f4_fma(float s, float4 a, float4 b) {
  return make_float4(fmaf(s, a.x, b.x), fmaf(s, a.y, b.y), fmaf(s, a.z, b.z), fmaf(s, a.w, b.w));
}
__device__ __forceinline__ float4 f4_scale(float s, float4 a) { return make_float4(s * a.x, s * a.y, s * a.z, s * a.w); }
__device__ __forceinline__ float4 f4_relu(float4 a) {
  return make_float4(fmaxf(a.x, 0.f), fmaxf(a.y, 0.f), fmaxf(a.z, 0.f), fmaxf(a.w, 0.f));
}
// streaming (read-once) and default loads of one 16-byte chunk
__device__ __forceinline__ float4 ld_f4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float4 ld_f4_stream(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void st_f4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void red_add_f4(float* p, float4 v) {
  atomicAdd(p + 0, v.x);
  atomicAdd(p + 1, v.y);
  atomicAdd(p + 2, v.z);
  atomicAdd(p + 3, v.w);
}

// ---- deterministic padding-row partials ------------------------------------------------------
// A gather backward adds every atom's share of its segment's padding row into that row.  In deterministic mode each "unit" (one atom slot of
// a CTA, which walks its atoms in increasing order and so meets the segments in increasing order) stores the partial of every padding row it
// meets, entry unit * jcap + j for the j-th row it meets, and tags the entry with the row; pad_rows_sum() then adds the entries of each row
// in entry order: CTA 0, 1, 2, ..., and inside a CTA slot 0, 1, 2, ...
struct PadParts {
  float* parts;     // [entries, ld]
  int* tags;        // [entries] padding row of the entry, -1 = unused
  int jcap;         // entries per unit
  long long entries;
};
// pad_parts_setup sizes jcap so that a unit never meets more rows than it has entries; should that bound ever fail, the unit's last entry is
// poisoned with NaN, so that its padding row's gradient shows the error instead of silently missing a partial.
__device__ __forceinline__ void pad_part_store(const PadParts& pp, long long unit, int& j, int pad_row, int ld, int c4, float4 v) {
  if (j < pp.jcap) {
    const long long e = unit * pp.jcap + j;
    st_f4(pp.parts + e * ld + c4, v);
    if (c4 == 0) pp.tags[e] = pad_row;
  } else {
    const float nan = __int_as_float(0x7fc00000);
    st_f4(pp.parts + (unit * pp.jcap + pp.jcap - 1) * ld + c4, make_float4(nan, nan, nan, nan));
  }
  ++j;
}

// ---- Philox4x32-7: counter-based dropout masks, regenerable from (seed, stream, index) -----
// Seven rounds is the smallest Philox4x32 variant that passes BigCrush (Salmon et al., SC'11, table 2; ten is the default safety margin).
// The masks are drawn in the GEMM epilogue, whose ALU work competes with the warps that feed the tensor core, so rounds are not free.
__device__ __forceinline__ uint4 philox4x32(uint64_t seed, uint64_t stream_id, uint64_t idx) {
  uint32_t k0 = static_cast<uint32_t>(seed), k1 = static_cast<uint32_t>(seed >> 32);
  uint32_t c0 = static_cast<uint32_t>(idx), c1 = static_cast<uint32_t>(idx >> 32);
  uint32_t c2 = static_cast<uint32_t>(stream_id), c3 = static_cast<uint32_t>(stream_id >> 32);
#pragma unroll
  for (int r = 0; r < 7; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}
// keep-mask scaling of 4 consecutive elements; idx4 = (linear element index) / 4
__device__ __forceinline__ float4 dropout4(float4 v, float p, float inv_keep, uint64_t seed, uint64_t stream_id, uint64_t idx4) {
  const uint4 r = philox4x32(seed, stream_id, idx4);
  const uint32_t thr = static_cast<uint32_t>(fminf(p, 1.f) * 4294967295.f);
  v.x = (r.x >= thr) ? v.x * inv_keep : 0.f;
  v.y = (r.y >= thr) ? v.y * inv_keep : 0.f;
  v.z = (r.z >= thr) ? v.z * inv_keep : 0.f;
  v.w = (r.w >= thr) ? v.w * inv_keep : 0.f;
  return v;
}

// ---- launchers shared between translation units ----------------------------------------------
int padded(int);
int bond_message_fwd(const rr_graph*, const float*, float*, int, int, cudaStream_t);
int bond_message_bwd(const rr_graph*, const float*, float*, int, cudaStream_t);
int neighbor_sum_fwd(const rr_graph*, int, const float*, float*, int, int, cudaStream_t);
int neighbor_sum_bwd(const rr_graph*, int, const float*, float*, int, cudaStream_t);
// gather backward + the ReLU / dropout backward that follows it (y: activation the mask comes from; acc_mode 0 none, 1 acc = dz, 2 acc += dz)
// det / det_bytes: scratch of deterministic mode (NULL: transient, see DetScratch)
int bond_message_bwd_act(const rr_graph*, const float* dpre, float* dm, int hp, const float* y, float scale, int preact, float* acc, int acc_mode,
                         int skip_out, cudaStream_t, void* det = nullptr, long long det_bytes = 0);
int neighbor_sum_bwd_act(const rr_graph*, int which, const float* dout, float* dsrc, int ld, const float* y, float scale, int preact, float* acc,
                         int acc_mode, int skip_out, cudaStream_t, void* det = nullptr, long long det_bytes = 0);
// det != NULL: the deterministic variant of a backward op, its padding-row partials carved from det (see PadParts)
int rowpipe_launch(int op, const rr_graph* g, int which, const float* src, float* out, int ld, int relu_src, const float* y, float scale, int preact,
                   float* acc, int acc_mode, int skip_out, cudaStream_t s, void* det = nullptr, long long det_bytes = 0, PadParts* pp = nullptr);
int pad_rows_act(float* out, const int* rows, int n_rows, int ld, const float* y, float scale, int preact, float* acc, int acc_mode, int skip_out,
                 cudaStream_t s);
// deterministic padding rows: bytes of scratch a gather backward over n_atoms rows of n_segments segments may need (either generation)
long long pad_parts_bytes(int n_atoms, int n_segments, int ld);
// carve the entries of `units` units of at most atoms_per_unit atoms out of scratch (RR_ERR_WORKSPACE when it is too small) and mark them unused
int pad_parts_setup(void* scratch, long long bytes, long long units, long long atoms_per_unit, int n_segments, int ld, PadParts* pp, cudaStream_t s);
// out[rows[r]] = sum of the entries tagged rows[r], in entry order
int pad_rows_sum(float* out, const int* rows, int n_rows, int ld, const PadParts& pp, cudaStream_t s);
// scratch for a deterministic launch: `given` when not NULL (RR_ERR_WORKSPACE if smaller than need), else cudaMallocAsync on s
int det_scratch(DetScratch* d, void* given, long long given_bytes, long long need, cudaStream_t s);
int readout_fwd(const rr_graph*, const float*, int, int, const float*, int, float*, int, float, uint64_t, uint64_t, cudaStream_t);
// p_vec: the FFN's dropout on vec, p_hid: the diff encoder's on hid
int readout_bwd(const rr_graph*, const float* dvec, int vp, const float* vec, const float* hid, float* dz, int hp, float p_vec, float p_hid,
                cudaStream_t);
int relu_bwd(long long, int, const float*, const float*, float, int, float*, float*, int, cudaStream_t);
int sub(long long, const float*, const float*, float*, cudaStream_t);
int sub_gather(long long rows, int ld, const float* a, const float* b, const int* map, float* out, cudaStream_t);
int scatter_add_rows(long long rows, int ld, const float* src, const int* map, float* dst, cudaStream_t);
int loss_fwdbwd(int, int, int, const float*, const float*, const int*, float, float, float*, float*, cudaStream_t, int max_group = 0);
int loss_max_group();
int rank_metrics(int, int, const float*, int, const double*, const int*, int, double, double*, cudaStream_t);
int rank_predict(int, int, int, const float*, long long, int, const int*, int, float*, cudaStream_t);
int graph_assemble(const rr_mol_store*, int, const int*, const int*, const int*, const int*, const int*, const int*, int, const int*, const int*,
                   const int*, const rr_graph*, cudaStream_t);
long long model_workspace_bytes(const rr_model_cfg_ex*, const rr_graph*, const rr_graph*);
long long model_buffer_offset(const rr_model_cfg_ex*, const rr_graph*, const rr_graph*, const char*);
int model_forward(const rr_model_cfg_ex*, const rr_params*, const rr_graph*, const rr_graph*, const float*, float*, void*, long long, cudaStream_t);
int model_backward(const rr_model_cfg_ex*, const rr_params*, const rr_graph*, const rr_graph*, const float*, rr_params*, void*, long long,
                   cudaStream_t);

// ---- dense layers (nn.Linear) ---------------------------------------------------------------------
// Pre-split images of fp32 weights for the tensor-core GEMMs: the images of the weight at base[i] are element i of each array.  The model
// makes them for its packed weights once per step (k_pack); rr_linear_dgrad_tc makes them for one transposed weight in caller scratch.
struct WeightImages {
  const float* base;
  float *tf32_hi, *tf32_lo;     // hi = w rounded to the nearest TF32 value, lo = w - hi
  uint16_t *bf16_hi, *bf16_lo;  // hi = bf16(w), lo = bf16(w - hi)
};

// Dispatch (rr_linear.cu): which kernel and operand split runs, from the precision switches and the shape.
// img: pre-split images of W1 / W2 (NULL: the tensor cores split the fp32 weights on chip).  pad_rows: the n_pad segment padding rows of Y,
// recomputed in exact arithmetic after a tensor-core forward (NULL: none).
int linear_fwd(int M, int n, const float* X1, int ldx1, const float* W1, int k1, const float* X2, int ldx2, const float* W2, int k2,
               const float* bias, const float* resid, int ldr, float* Y, int ldy, int flags, float p, uint64_t seed, uint64_t stream_id,
               cudaStream_t s, const WeightImages* img = nullptr, const int* pad_rows = nullptr, int n_pad = 0);
// dX[M, k] (+)= dZ[M, n] W[n, k]; the tensor cores read the images of the transposed copy Wt[k, ldwt], the SIMT kernel reads W
int linear_dgrad(int M, int n, int k, const float* dZ, int lddz, const float* W, int ldw, const float* Wt, int ldwt, float* dX, int lddx,
                 int accumulate, const WeightImages& img, cudaStream_t s);
int linear_dgrad_tc(int M, int n, int k, const float* dZ, int lddz, const float* W, int ldw, float* dX, int lddx, int accumulate, void* scratch,
                    long long scratch_bytes, cudaStream_t s);
int linear_wgrad(int, int, int, const float*, int, const float*, int, float*, int, float*, cudaStream_t, void* det = nullptr, long long det_bytes = 0);
// deterministic mode: bytes of scratch linear_wgrad(M, n, k, ...) needs (row-slab partials of dW and of the bias gradient), any GEMM mode
long long wgrad_det_bytes(int M, int n, int k);
// dbias[n] += colsum(dZ[M, n]) over every row, for a bias whose weight is frozen: row slabs store partials, a second pass adds them in slab
// order (no atomics, the same bits on every run in both modes).  Scratch: det when given (>= bias_grad_bytes(M, n)), else transient.
int linear_bias_grad(int M, int n, const float* dZ, int lddz, float* dbias, cudaStream_t s, void* det = nullptr, long long det_bytes = 0);
long long bias_grad_bytes(int M, int n);

// fp32 SIMT launchers (rr_gemm_simt.cu)
int simt_fwd(int M, int n, const float* X1, int ldx1, const float* W1, int k1, const float* X2, int ldx2, const float* W2, int k2, const float* bias,
             const float* resid, int ldr, float* Y, int ldy, int flags, float p, uint64_t seed, uint64_t stream_id, cudaStream_t s);
int simt_dgrad(int M, int n, int k, const float* dZ, int lddz, const float* W, int ldw, float* dX, int lddx, int accumulate, cudaStream_t s);
// Weight gradient, split over row slabs of the M reduction rows (its arguments checked by the caller).
// slab != NULL (deterministic mode): slab z of the reduction stores its dW tile to slab + z * n * k (row stride k) and, when dbias != NULL,
// its bias partial to slab + splits * n * k + z * n, instead of adding into dW / dbias; *splits receives the slab count.  The same holds
// for tc_wgrad.
int simt_wgrad(int M, int n, int k, const float* dZ, int lddz, const float* X, int ldx, float* dW, int lddw, float* dbias, cudaStream_t s,
               float* slab = nullptr, int* splits = nullptr);
int simt_wgrad_splits(int M, int n, int k, int* chunk);

// tcgen05 launchers (rr_gemm_tc.cu).  The B operand of the forward / dgrad GEMM (the weights W[n, K], row stride ldw elements) arrives as
enum TcSplit {
  TC_FP32,       // the fp32 weights (hi), split into TF32 (hi, lo) on chip
  TC_TF32_PAIR,  // TF32 images: hi and lo are float
  TC_BF16_PAIR,  // bf16 images: hi and lo are uint16_t, 3 x bf16 products
};
struct TcSrc {    // one source of the K reduction: X[M, K] (row stride ldx floats) times W^T
  const float* X;
  int ldx;
  const void *hi, *lo;
  int ldw, K;
};
bool tc_supported(int M, int n, int k1, int k2, int ldx1, int ldx2);
bool tc_linear_bf16_supported(int M, int n, int k, int ldx, int ldw);
// Y[M, n] = epi(sum over the nsrc sources of X W^T) on k_tc_gemm2
int tc_linear(TcSplit split, int M, int n, const TcSrc* src, int nsrc, const float* bias, const float* resid, int ldr, float* Y, int ldy, int relu,
              int accumulate, float p, uint64_t seed, uint64_t stream_id, int kclass, cudaStream_t s);
// rr_linear_dgrad_tc: layout of the images of Wt = W[n, k]^T (row stride *ldt) in caller scratch, and the kernel that fills it
long long tc_dgrad_scratch_bytes(int n, int k);
WeightImages tc_dgrad_images(int n, int k, void* scratch, int* ldt);
int tc_transpose_split(const float* W, int n, int k, int ldw, const WeightImages& img, int ldt, cudaStream_t s);
bool tc_wgrad_supported(int M, int n, int k, int lddz, int ldx);
// bf16: 3 x bf16 products (k_tc_wgrad3), else 3 x TF32 (k_tc_wgrad2)
int tc_wgrad(bool bf16, int M, int n, int k, const float* dZ, int lddz, const float* X, int ldx, float* dW, int lddw, float* dbias, cudaStream_t s,
             float* slab = nullptr, int* splits = nullptr);
// slab count of tc_wgrad with slabs of whole stages of stage_rows rows (*chunk rows each); stage_rows = 0: the upper bound over every stage
// height, which sizes the deterministic scratch
int tc_wgrad_splits(int M, int n, int k, int stage_rows = 0, int* chunk = nullptr);

}  // namespace rr
