// Dense layers (the nn.Linear call sites of mpn.py / base_model.py): the one place that decides which GEMM kernel and which operand split
// run.  rr_gemm_simt.cu and rr_gemm_tc.cu only launch what is decided here.
//
// Policy by gemm mode (rr_set_gemm_mode).  TC = the tcgen05 kernels where the shape and the alignment suit them, the SIMT kernels otherwise.
//
//   mode | forward | dgrad of rr_model_backward | wgrad           | padding-row fix-up after the forward
//   -----+---------+----------------------------+-----------------+-------------------------------------
//    0   | SIMT    | SIMT                       | SIMT            | no
//    1   | TC      | TC                         | TC for M >= 256 | yes
//    2   | TC      | SIMT                       | SIMT            | yes
//    3   | SIMT    | TC                         | SIMT            | no
//
//   - rr_linear_dgrad is SIMT in every mode; rr_linear_dgrad_tc is TC in every mode (RR_ERR_UNSUPPORTED for a shape it does not suit).
//   - The fix-up runs after every forward that names padding rows (the model's), in modes 1 and 2, also when the shape fell back to SIMT.
//   - Operand split of a TC forward: 3 x bf16 when rr_set_forward_bf16(1) and the caller has weight images (the model), else 3 x TF32, from
//     the caller's images or split on chip (rr_linear_fwd).  Of a TC dgrad and wgrad: 3 x bf16 when rr_set_backward_bf16(1) (the default),
//     else 3 x TF32 (the wgrad's k_tc_wgrad2).  A shape the bf16 forward / dgrad refuses takes the TF32 kernel.
//   - Deterministic mode changes none of these choices: the wgrad's row slabs store their partials and k_wgrad_slab_sum adds them in order.
//   - A bias gradient without its weight's (rr_model_backward with the weight frozen) is linear_bias_grad, fp32 SIMT in every mode.
#include "rr_common.cuh"

namespace rr {

// One source of a tensor-core GEMM in the given split: W itself (TC_FP32) or its images in img
static TcSrc tc_src(TcSplit split, const WeightImages* img, const float* X, int ldx, const float* W, int ldw, int K) {
  if (split == TC_FP32) return {X, ldx, W, nullptr, ldw, K};
  const ptrdiff_t i = W - img->base;
  if (split == TC_BF16_PAIR) return {X, ldx, img->bf16_hi + i, img->bf16_lo + i, ldw, K};
  return {X, ldx, img->tf32_hi + i, img->tf32_lo + i, ldw, K};
}

// ---- padding rows in exact arithmetic -------------------------------------------------------
// A segment's padding bond / padding atom row is gathered by EVERY padded neighbour slot of the segment (featurization.py:281-286), so in
// the backward pass it collects the gradient of all of them: at the c5 batch one such row weighs as much as ~10^5 ordinary rows.  Its ReLU
// masks must therefore be decided as the reference's fp32 run decides them.  The tensor-core forward (3 x TF32, RZ accumulation) leaves
// 2-5e-6 of relative error on a pre-activation, which flips the mask of an entry that lies that close to zero; on an ordinary row such a
// flip moves the gradient by one row's share, on a padding row by a macroscopic amount.  After every tensor-core forward GEMM whose output
// feeds a ReLU, the n_segments padding rows are therefore recomputed here from the unsplit fp32 weights with fp64 accumulation (one
// rounding, tighter than any fp32 GEMM) and overwritten, epilogue (bias, residual, ReLU, the same Philox dropout mask) included.
struct PadFix {
  const int* rows;
  int n_rows, n;
  const float *X1, *W1, *X2, *W2, *bias, *resid;
  int ldx1, k1, ldx2, k2, ldr;
  float* Y;
  int ldy, relu;
  float p, inv_keep;
  uint64_t seed, stream_id;
};
// One warp per output column (grid = rows x ceil(n / 8), 8 warps per block): the k loop is unrolled into independent loads and four
// fp64 partial sums, so a launch is a couple of microseconds (the first version, one warp per ~5 columns with a serial chain, took 20).
__device__ __forceinline__ double pad_dot(const float* __restrict__ x, const float* __restrict__ w, int k, int lane) {
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
  int i = lane;
  for (; i + 96 < k; i += 128) {
    const float x0 = x[i], x1 = x[i + 32], x2 = x[i + 64], x3 = x[i + 96];
    const float w0 = __ldg(w + i), w1 = __ldg(w + i + 32), w2 = __ldg(w + i + 64), w3 = __ldg(w + i + 96);
    a0 = fma(static_cast<double>(x0), static_cast<double>(w0), a0);
    a1 = fma(static_cast<double>(x1), static_cast<double>(w1), a1);
    a2 = fma(static_cast<double>(x2), static_cast<double>(w2), a2);
    a3 = fma(static_cast<double>(x3), static_cast<double>(w3), a3);
  }
  for (; i < k; i += 32) a0 = fma(static_cast<double>(x[i]), static_cast<double>(__ldg(w + i)), a0);
  return (a0 + a1) + (a2 + a3);
}
__global__ void __launch_bounds__(256) k_pad_rows_linear(PadFix a) {
  const size_t row = static_cast<size_t>(__ldg(a.rows + blockIdx.x));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = blockIdx.y * 8 + warp;
  if (c >= a.n) return;
  double acc = pad_dot(a.X1 + row * a.ldx1, a.W1 + static_cast<size_t>(c) * a.k1, a.k1, lane);
  if (a.X2) acc += pad_dot(a.X2 + row * a.ldx2, a.W2 + static_cast<size_t>(c) * a.k2, a.k2, lane);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) {
    if (a.bias) acc += static_cast<double>(a.bias[c]);
    if (a.resid) acc += static_cast<double>(a.resid[row * a.ldr + c]);
    float o = static_cast<float>(acc);
    if (a.relu) o = fmaxf(o, 0.f);
    if (a.p > 0.f) {   // element (c & 3) of the 4-wide Philox draw the GEMM epilogue makes for this chunk (dropout4)
      const uint4 r = philox4x32(a.seed, a.stream_id, (row * a.ldy + c) >> 2);
      const uint32_t thr = static_cast<uint32_t>(fminf(a.p, 1.f) * 4294967295.f);
      const uint32_t rv = (c & 3) == 0 ? r.x : ((c & 3) == 1 ? r.y : ((c & 3) == 2 ? r.z : r.w));
      o = rv >= thr ? o * a.inv_keep : 0.f;
    }
    a.Y[row * a.ldy + c] = o;
  }
}
// same argument order as linear_fwd; W1 / W2 are the raw (unsplit) weights
static int pad_rows_linear(const int* rows, int n_rows, int n, const float* X1, int ldx1, const float* W1, int k1, const float* X2, int ldx2, const float* W2,
                           int k2, const float* bias, const float* resid, int ldr, float* Y, int ldy, int flags, float p, uint64_t seed,
                           uint64_t stream_id, cudaStream_t s) {
  if (n_rows <= 0 || rows == nullptr) return RR_OK;
  ProfScope prof_scope(KC_MISC, s);
  PadFix a{};
  a.rows = rows;
  a.n_rows = n_rows;
  a.n = n;
  a.X1 = X1; a.ldx1 = ldx1; a.W1 = W1; a.k1 = k1;
  a.X2 = (X2 && k2 > 0) ? X2 : nullptr; a.ldx2 = ldx2; a.W2 = W2; a.k2 = k2;
  a.bias = bias; a.resid = resid; a.ldr = ldr;
  a.Y = Y; a.ldy = ldy;
  a.relu = flags & 1;
  a.p = (flags & 2) ? p : 0.f;
  a.inv_keep = a.p > 0.f ? 1.f / (1.f - a.p) : 1.f;
  a.seed = seed;
  a.stream_id = stream_id;
  k_pad_rows_linear<<<dim3(n_rows, (n + 7) / 8), 256, 0, s>>>(a);
  RR_LAUNCH_CHECK("k_pad_rows_linear");
  return RR_OK;
}

// ---- forward ------------------------------------------------------------------------------------
int linear_fwd(int M, int n, const float* X1, int ldx1, const float* W1, int k1, const float* X2, int ldx2, const float* W2, int k2,
               const float* bias, const float* resid, int ldr, float* Y, int ldy, int flags, float p, uint64_t seed, uint64_t stream_id,
               cudaStream_t s, const WeightImages* img, const int* pad_rows, int n_pad) {
  const int mode = g_gemm_mode.load();
  const bool tc = mode == 1 || mode == 2;
  const bool two = X2 && k2 > 0;
  // what every tensor-core forward needs of the activations and the epilogue operands
  const bool tc_operands = tc && aligned16(X1) && aligned16(Y) && (!resid || (aligned16(resid) && (ldr & 3) == 0)) && (!bias || aligned16(bias)) &&
                           (ldy & 3) == 0 && p >= 0.f && p < 1.f;
  bool on_tc = true;
  TcSplit split = TC_FP32;
  if (tc_operands && img && g_fwd_bf16.load() && tc_linear_bf16_supported(M, n, k1, ldx1, k1) &&
      (!two || (tc_linear_bf16_supported(M, n, k2, ldx2, k2) && aligned16(X2))))
    split = TC_BF16_PAIR;
  else if (tc_operands && tc_supported(M, n, k1, X2 ? k2 : 0, ldx1, X2 ? ldx2 : 0) && aligned16(W1) && (!X2 || (aligned16(X2) && aligned16(W2))))
    split = img ? TC_TF32_PAIR : TC_FP32;
  else
    on_tc = false;
  if (on_tc) {
    const TcSrc src[2] = {tc_src(split, img, X1, ldx1, W1, k1, k1), two ? tc_src(split, img, X2, ldx2, W2, k2, k2) : TcSrc{}};
    RR_TRY(tc_linear(split, M, n, src, two ? 2 : 1, bias, resid, ldr, Y, ldy, flags & 1, 0, (flags & 2) ? p : 0.f, seed, stream_id, KC_GEMM_FWD, s));
  } else {
    RR_TRY(simt_fwd(M, n, X1, ldx1, W1, k1, X2, ldx2, W2, k2, bias, resid, ldr, Y, ldy, flags, p, seed, stream_id, s));
  }
  if (tc) RR_TRY(pad_rows_linear(pad_rows, n_pad, n, X1, ldx1, W1, k1, X2, ldx2, W2, k2, bias, resid, ldr, Y, ldy, flags, p, seed, stream_id, s));
  return RR_OK;
}

// ---- dgrad --------------------------------------------------------------------------------------
// operand split of a tensor-core dgrad dX[M, k] = dZ[M, n] Wt[k, ldwt]^T; false when the shape does not suit the kernel
static bool dgrad_split(int M, int n, int k, int lddz, int ldwt, TcSplit* split) {
  *split = g_bwd_bf16.load() && tc_linear_bf16_supported(M, k, n, lddz, ldwt) ? TC_BF16_PAIR : TC_TF32_PAIR;
  return *split == TC_BF16_PAIR || tc_supported(M, k, n, 0, lddz, 0);
}
static int dgrad_tc(TcSplit split, int M, int n, int k, const float* dZ, int lddz, const float* Wt, int ldwt, float* dX, int lddx, int accumulate,
                    const WeightImages& img, cudaStream_t s) {
  const TcSrc src = tc_src(split, &img, dZ, lddz, Wt, ldwt, n);
  return tc_linear(split, M, k, &src, 1, nullptr, nullptr, 0, dX, lddx, 0, accumulate, 0.f, 0, 0, KC_GEMM_DGRAD, s);
}

int linear_dgrad(int M, int n, int k, const float* dZ, int lddz, const float* W, int ldw, const float* Wt, int ldwt, float* dX, int lddx,
                 int accumulate, const WeightImages& img, cudaStream_t s) {
  const int mode = g_gemm_mode.load();
  TcSplit split;
  if ((mode == 1 || mode == 3) && dgrad_split(M, n, k, lddz, ldwt, &split)) return dgrad_tc(split, M, n, k, dZ, lddz, Wt, ldwt, dX, lddx, accumulate, img, s);
  return simt_dgrad(M, n, k, dZ, lddz, W, ldw, dX, lddx, accumulate, s);
}

int linear_dgrad_tc(int M, int n, int k, const float* dZ, int lddz, const float* W, int ldw, float* dX, int lddx, int accumulate, void* scratch,
                    long long scratch_bytes, cudaStream_t s) {
  RR_REQUIRE(M > 0 && n > 0 && k > 0 && dZ && W && dX && scratch, "linear_dgrad_tc: bad argument");
  RR_REQUIRE(aligned16(dZ) && aligned16(dX) && aligned16(scratch) && !(lddz & 3) && !(lddx & 3), "linear_dgrad_tc: operands must be 16-byte aligned rows");
  RR_REQUIRE(scratch_bytes >= tc_dgrad_scratch_bytes(n, k), "linear_dgrad_tc: scratch %lld bytes < required %lld", scratch_bytes, tc_dgrad_scratch_bytes(n, k));
  int ldt = 0;
  const WeightImages img = tc_dgrad_images(n, k, scratch, &ldt);
  TcSplit split;
  if (!dgrad_split(M, n, k, lddz, ldt, &split)) return fail(RR_ERR_UNSUPPORTED, "linear_dgrad_tc: shape M %d n %d k %d does not suit the tensor-core kernel (k %% 16, n %% 4)", M, n, k);
  RR_TRY(tc_transpose_split(W, n, k, ldw, img, ldt, s));
  return dgrad_tc(split, M, n, k, dZ, lddz, img.base, ldt, dX, lddx, accumulate, img, s);
}

// ---- wgrad --------------------------------------------------------------------------------------
long long wgrad_det_bytes(int M, int n, int k) {
  if (M <= 0 || n <= 0 || k <= 0) return 0;
  const int tcs = tc_wgrad_splits(M, n, k), simt = simt_wgrad_splits(M, n, k, nullptr);
  const long long splits = tcs > simt ? tcs : simt;
  return splits * (static_cast<long long>(n) * k + n) * static_cast<long long>(sizeof(float));
}

// dW[i, j] += sum over z = 0, 1, 2, ... of slab[z][i, j];  dbias[i] += the same over the bias partials
__global__ void k_wgrad_slab_sum(int n, int k, int splits, const float* __restrict__ slab, const float* __restrict__ slab_bias, float* __restrict__ dW,
                                 int lddw, float* __restrict__ dbias) {
  const int k4 = k >> 2;
  const long long plane = static_cast<long long>(n) * k;
  const long long total = static_cast<long long>(n) * k4;
  for (long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; t < total + n; t += static_cast<long long>(gridDim.x) * blockDim.x) {
    if (t < total) {
      const int i = static_cast<int>(t / k4), j = static_cast<int>(t - static_cast<long long>(i) * k4) << 2;
      const float* p = slab + static_cast<long long>(i) * k + j;
      float4 acc = ld_f4(p);
#pragma unroll 8
      for (int z = 1; z < splits; ++z) acc = f4_add(acc, ld_f4(p + z * plane));
      float* d = dW + static_cast<size_t>(i) * lddw + j;
      st_f4(d, f4_add(*reinterpret_cast<const float4*>(d), acc));
    } else if (dbias) {
      const int i = static_cast<int>(t - total);
      float acc = slab_bias[i];
      for (int z = 1; z < splits; ++z) acc += slab_bias[static_cast<long long>(z) * n + i];
      dbias[i] += acc;
    }
  }
}

int linear_wgrad(int M, int n, int k, const float* dZ, int lddz, const float* X, int ldx, float* dW, int lddw, float* dbias, cudaStream_t s, void* det,
                 long long det_bytes) {
  RR_REQUIRE(M >= 0 && n > 0 && k > 0 && (n & 3) == 0 && (k & 3) == 0, "linear_wgrad: M %d n %d k %d", M, n, k);
  RR_TRY(check_mat("dZ", dZ, lddz));
  RR_TRY(check_mat("X", X, ldx));
  RR_TRY(check_mat("dW", dW, lddw));
  if (M == 0) return RR_OK;
  const bool tc = g_gemm_mode.load() == 1 && M >= 256 && tc_wgrad_supported(M, n, k, lddz, ldx);
  const bool bf16 = g_bwd_bf16.load() != 0;
  if (!deterministic()) {
    if (tc) return tc_wgrad(bf16, M, n, k, dZ, lddz, X, ldx, dW, lddw, dbias, s);
    return simt_wgrad(M, n, k, dZ, lddz, X, ldx, dW, lddw, dbias, s);
  }
  // Deterministic: every row slab stores its partial dW tile (and bias partial) to scratch, then k_wgrad_slab_sum adds them in slab order.
  DetScratch ds;
  RR_TRY(det_scratch(&ds, det, det_bytes, wgrad_det_bytes(M, n, k), s));
  float* slab = static_cast<float*>(ds.p);
  int splits = 0;
  if (tc) RR_TRY(tc_wgrad(bf16, M, n, k, dZ, lddz, X, ldx, dW, lddw, dbias, s, slab, &splits));
  else RR_TRY(simt_wgrad(M, n, k, dZ, lddz, X, ldx, dW, lddw, dbias, s, slab, &splits));
  ProfScope prof_scope(KC_GEMM_WGRAD, s);
  const long long work = static_cast<long long>(n) * (k >> 2) + n;
  long long blocks = (work + 255) / 256;
  if (blocks > num_sms() * 8) blocks = num_sms() * 8;
  k_wgrad_slab_sum<<<static_cast<int>(blocks), 256, 0, s>>>(n, k, splits, slab, slab + splits * static_cast<long long>(n) * k, dW, lddw, dbias);
  RR_LAUNCH_CHECK("k_wgrad_slab_sum");
  return RR_OK;
}

// ---- bias gradient alone -------------------------------------------------------------------------
// The column sum of dZ over all M rows, padding rows included, as the weight gradient's fused bias partial takes it; not the same bits.
// Slab z of rows_per_slab rows: a (32 x 8) block sums 32 float4 columns over its rows, eight row lanes reduced in lane order, and stores the
// partial to part[z * n ..]; k_bias_colsum_total adds the partials of each column in slab order.
__global__ void __launch_bounds__(256) k_bias_colsum_slabs(int M, int n, int rows_per_slab, const float* __restrict__ dZ, int lddz,
                                                           float* __restrict__ part) {
  __shared__ float4 red[8][32];
  const int c = (blockIdx.y * 32 + threadIdx.x) * 4;
  const long long r0 = static_cast<long long>(blockIdx.x) * rows_per_slab;
  const long long r1 = r0 + rows_per_slab < M ? r0 + rows_per_slab : M;
  float4 acc = f4_zero();
  if (c < n)
    for (long long r = r0 + threadIdx.y; r < r1; r += 8) acc = f4_add(acc, ld_f4(dZ + r * lddz + c));
  red[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && c < n) {
#pragma unroll
    for (int y = 1; y < 8; ++y) acc = f4_add(acc, red[y][threadIdx.x]);
    st_f4(part + static_cast<long long>(blockIdx.x) * n + c, acc);
  }
}
__global__ void k_bias_colsum_total(int n, int slabs, const float* __restrict__ part, float* __restrict__ dbias) {
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < n; c += gridDim.x * blockDim.x) {
    float acc = part[c];
    for (int z = 1; z < slabs; ++z) acc += part[static_cast<long long>(z) * n + c];
    dbias[c] += acc;
  }
}

// slab height: at least 64 rows, at most 2 slabs per SM; a multiple of the 8 row lanes
static int bias_grad_rows_per_slab(int M) {
  const int per = (M + 2 * num_sms() - 1) / (2 * num_sms());
  return ((per > 64 ? per : 64) + 7) / 8 * 8;
}
long long bias_grad_bytes(int M, int n) {
  if (M <= 0 || n <= 0) return 0;
  const int rows = bias_grad_rows_per_slab(M);
  return static_cast<long long>((M + rows - 1) / rows) * n * static_cast<long long>(sizeof(float));
}

int linear_bias_grad(int M, int n, const float* dZ, int lddz, float* dbias, cudaStream_t s, void* det, long long det_bytes) {
  RR_REQUIRE(M >= 0 && n > 0 && (n & 3) == 0, "linear_bias_grad: M %d n %d", M, n);
  RR_TRY(check_mat("dZ", dZ, lddz));
  RR_REQUIRE(dbias != nullptr, "linear_bias_grad: dbias is NULL");
  if (M == 0) return RR_OK;
  const int rows = bias_grad_rows_per_slab(M), slabs = (M + rows - 1) / rows;
  DetScratch ds;
  RR_TRY(det_scratch(&ds, det, det_bytes, bias_grad_bytes(M, n), s));
  float* part = static_cast<float*>(ds.p);
  {
    ProfScope prof_scope(KC_GEMM_WGRAD, s);
    k_bias_colsum_slabs<<<dim3(slabs, (n / 4 + 31) / 32), dim3(32, 8), 0, s>>>(M, n, rows, dZ, lddz, part);
    RR_LAUNCH_CHECK("k_bias_colsum_slabs");
  }
  ProfScope prof_scope(KC_GEMM_WGRAD, s);
  k_bias_colsum_total<<<(n + 255) / 256, 256, 0, s>>>(n, slabs, part, dbias);
  RR_LAUNCH_CHECK("k_bias_colsum_total");
  return RR_OK;
}

}  // namespace rr
